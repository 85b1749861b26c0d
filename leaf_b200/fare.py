"""The LEAF / TextFARE training iteration on the engine: the body of train_one_epoch_text_only's batch loop
(/root/reference/utils_AT.py:291-366) - frozen anchor, LEAF attack, forward + backward of the B winners, gradient
accumulation, clipping, AdamW with the reference's two parameter groups (/root/reference/train_AT_text_only.py:326-341)
and, under torch.distributed, the data-parallel gradient all-reduce the reference delegates to DDP.

What is native: everything that touches the tower (K1-K4), the AdamW update (one launch over the flat parameter
buffer), the gradient-norm reduction. What stays torch: the two-line loss expression and the NCCL all-reduce call.
The scheduler, the data loader and logging are the caller's, unchanged (SURVEY.md 8: out of scope). Checkpoints cover the
trainer's own state (FareTrainer.state_dict / load_state_dict, which resume bit for bit) and the reference's epoch checkpoint
format (FareTrainer.reference_checkpoint / load_reference_checkpoint, train_AT_text_only.py:351-372, 516-525, 560-569).
"""
from __future__ import annotations

import contextlib
import math
import os
import weakref

import numpy as np
import torch
import torch.distributed as dist

from .attack import V_DEFAULT, attack_text_leaf
from .eval_attacks import attack_text_charmer_inference
from .tower import LeafTextTower, no_weight_decay, text_tower_state_dict

STATE_FORMAT, STATE_VERSION = "leaf_b200.FareTrainer", 1


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

            tower.leaf_engine.set_backward_hook(thunk)

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
        eng.sumsq(g, self._norm)
        total = math.sqrt(float(self._norm.item())) * grad_scale
        return min(1.0, self.grad_clip_norm / (total + 1e-6))

    def optimizer_step(self, grad_scale: float = 1.0):
        """utils_AT.py:338-362 with scaler = None: all-reduce (DDP's job in the reference), clip, AdamW, zero_grad; then the
        engine re-casts its bf16 operand copies from the updated fp32 parameters."""
        t = self.tower
        self._exchange()
        scale = grad_scale
        if self.grad_clip_norm is not None:                       # the clip is folded into AdamW's gradient scale
            scale *= self._clip_scale(grad_scale)
        self.opt_step += 1
        t.leaf_engine.adamw(t.flat_params, t.flat_grads, self.exp_avg, self.exp_avg_sq, n_nodecay=t.n_nodecay,
                            lr=self.lr_at(self.opt_step), beta1=self.beta1, beta2=self.beta2, eps=self.eps, weight_decay=self.wd,
                            step=self.opt_step, grad_scale=scale)
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
        with t.leaf_engine.sm_budget(self.backward_sm_budget) if budget else contextlib.nullcontext():
            (loss / self.accum_freq).backward()                                            # :329-337
        if self.overlap_allreduce:
            self._hook_armed = False
        self.micro += 1
        if last:
            self.optimizer_step()
        elif clip_now:
            self._exchange()                                  # averaging identical accumulated values again changes nothing
            s = self._clip_scale()
            if s < 1.0:
                t.leaf_engine.scale(t.flat_grads, s)
        return loss.detach(), adv_texts

    # ---- checkpoints -----------------------------------------------------------------------------------------------------
    def _check_idle(self, what):
        if self._works:
            raise RuntimeError(f"FareTrainer.{what}() is only legal between step() calls: {len(self._works)} gradient all-reduces "
                               "of the overlapped exchange are still outstanding")

    def _config(self):
        e = self.tower.leaf_engine
        return {"width": e.width, "layers": e.layers, "heads": e.heads, "embed_dim": e.embed_dim, "quick_gelu": e.quick_gelu}

    def _by_name(self, flat):
        """{open_clip name: view} of a buffer laid out like the tower's flat parameters (the alignment padding left out)."""
        return {k: flat[off:off + n].view(shape) for k, (off, n, shape) in self.tower._slices.items()}

    def state_dict(self, include_rng: bool = True) -> dict:
        """Everything a resumed run needs to continue this one bit for bit (under torch.use_deterministic_algorithms): the
        trained tower's parameters, both AdamW moments, the counters, the gradients accumulated so far in an unfinished
        accumulation window, and (include_rng) the global numpy RNG the attack draws from, which the reference does not save.
        Tensors are keyed by open_clip name, not flat offset; they are views of the live buffers (as nn.Module.state_dict's
        are), so torch.save them, or clone them, before the next step(). The dict holds tensors, numbers, strings and
        lists only, so torch.load(weights_only=True) reads it back.

        Not included: the frozen anchor tower (the pretrained model; the caller rebuilds it, as the reference does), the
        caller's LR scheduler and data position. Under torchrun every rank holds the same parameters and moments but its own
        numpy RNG stream (seed + rank): either every rank saves its own state_dict(), or rank 0 saves the whole state and every
        rank saves its state_dict()["numpy_rng"] and puts it back into rank 0's state before load_state_dict. Only legal
        between step() calls."""
        self._check_idle("state_dict")
        t = self.tower
        rng = None
        if include_rng:
            name, key, pos, has_gauss, gauss = np.random.get_state()
            rng = (name, key.tolist(), int(pos), int(has_gauss), float(gauss))
        hparams = dict(V=[int(c) for c in self.V], rho=self.rho, k_adv=self.k_adv, lr=self.lr, wd=self.wd, beta1=self.beta1,
                       beta2=self.beta2, eps=self.eps, accum_freq=self.accum_freq, grad_clip_norm=self.grad_clip_norm,
                       constrain=self.constrain if isinstance(self.constrain, bool) else "callable",
                       normalize_fare=self.normalize_fare, use_charmer=self.use_charmer)
        return {"format": STATE_FORMAT, "version": STATE_VERSION, "config": self._config(), "hparams": hparams,
                "opt_step": self.opt_step, "micro": self.micro,
                "params": self._by_name(t.flat_params), "exp_avg": self._by_name(self.exp_avg),
                "exp_avg_sq": self._by_name(self.exp_avg_sq),
                "grads": self._by_name(t.flat_grads) if self.micro % self.accum_freq else None,   # zero between windows
                "numpy_rng": rng}

    def load_state_dict(self, state: dict):
        """Restore a state_dict(): the tower shape and every tensor's name and shape are checked first (ValueError naming each
        mismatch, nothing changed); then the values are copied INTO the existing buffers, so the .grad views, the backward
        hook's ranges and the engine binding stay valid, the counters and (when saved) the numpy RNG are restored and the
        engine re-casts its operand copies. The hyper-parameters are this trainer's own: the state records them but a
        resumed run may change them. Only legal between step() calls."""
        self._check_idle("load_state_dict")
        if state.get("format") != STATE_FORMAT or state.get("version") != STATE_VERSION:
            raise ValueError(f"not a FareTrainer state: format {state.get('format')!r} version {state.get('version')!r}, "
                             f"expected {STATE_FORMAT!r} version {STATE_VERSION}")
        bad = [f"config {k}: {state['config'].get(k)!r} in the state, {v!r} here" for k, v in self._config().items()
               if state["config"].get(k) != v]
        slices = self.tower._slices
        for group in ("params", "exp_avg", "exp_avg_sq", "grads"):
            named = state[group]
            if named is None:
                continue
            bad += [f"{group}: missing {k}" for k in slices if k not in named]
            bad += [f"{group}: unexpected {k}" for k in named if k not in slices]
            bad += [f"{group}: shape of {k} {tuple(v.shape)}, here {slices[k][2]}" for k, v in named.items()
                    if k in slices and tuple(v.shape) != slices[k][2]]
        if (state["grads"] is not None) != bool(state["micro"] % self.accum_freq):
            bad.append(f"accumulation window: micro-batch {state['micro']} with accum_freq {self.accum_freq}, and the state "
                       f"{'has' if state['grads'] is not None else 'has no'} pending gradients")
        if bad:
            raise ValueError("FareTrainer state does not fit this trainer: " + "; ".join(bad))
        with torch.no_grad():
            for group, flat in (("exp_avg", self.exp_avg), ("exp_avg_sq", self.exp_avg_sq), ("grads", self.tower.flat_grads)):
                if state[group] is None:
                    flat.zero_()
                    continue
                for k, view in self._by_name(flat).items():
                    view.copy_(state[group][k])
        self.tower.load_open_clip_state_dict(state["params"])                 # copies in place and refreshes the engine
        self.opt_step, self.micro = int(state["opt_step"]), int(state["micro"])
        if state.get("numpy_rng") is not None:
            name, key, pos, has_gauss, gauss = state["numpy_rng"]
            np.random.set_state((name, np.asarray(key, dtype=np.uint32), int(pos), int(has_gauss), float(gauss)))

    def _reference_groups(self, model):
        """The parameters of the reference's two AdamW groups (train_AT_text_only.py:326-341): model.named_parameters() in
        order, split by the reference's exclude rule, all of them whatever their requires_grad now (the reference builds its
        optimizer before it freezes the visual tower, SURVEY.md appendix F #9); and {id(parameter): open_clip name} of the
        text-tower parameters among them, checked against the trained tower."""
        named = list(model.named_parameters())
        groups = ([p for n, p in named if no_weight_decay(n, p.dim())], [p for n, p in named if not no_weight_decay(n, p.dim())])
        text = text_tower_state_dict(dict(named))
        slices = self.tower._slices
        bad = [f"missing from the model: {k}" for k in slices if k not in text]
        bad += [f"not in the trained tower: {k}" for k in text if k not in slices]
        bad += [f"shape of {k}: {tuple(p.shape)} in the model, {slices[k][2]} in the trained tower" for k, p in text.items()
                if k in slices and tuple(p.shape) != slices[k][2]]
        if bad:
            raise ValueError("the model's text tower does not match the trained one: " + "; ".join(bad))
        return groups, {id(p): k for k, p in text.items()}

    def reference_checkpoint(self, model, epoch: int, name: str) -> dict:
        """The dict the reference saves every epoch (train_AT_text_only.py:516-525, 560-569), for `model`, the caller's open_clip
        CLIP (or its DDP wrapper): "state_dict" is model.state_dict() with its text-tower entries replaced by the trained
        tower's (the model's own key prefixes are kept; the visual tower and logit_scale pass through), "optimizer" the
        state_dict() of a torch.optim.AdamW over the reference's two parameter groups holding this trainer's step and
        moments for the text parameters (the others have no state, as in the reference). There is no "scaler" entry: the
        engine trains in bf16 without a GradScaler. Tensors are views of the live buffers; torch.save before the next step()."""
        self._check_idle("reference_checkpoint")
        groups, text = self._reference_groups(model)
        params, m, v = self._by_name(self.tower.flat_params), self._by_name(self.exp_avg), self._by_name(self.exp_avg_sq)
        sd = model.state_dict()
        for k, key in text_tower_state_dict({key: key for key in sd}).items():
            sd[key] = params[k]
        opt = torch.optim.AdamW([{"params": groups[0], "weight_decay": 0.0}, {"params": groups[1], "weight_decay": self.wd}],
                                lr=self.lr, betas=(self.beta1, self.beta2), eps=self.eps)
        if self.opt_step:
            for p in groups[0] + groups[1]:
                k = text.get(id(p))
                if k is not None:
                    opt.state[p] = {"step": torch.tensor(float(self.opt_step)), "exp_avg": m[k], "exp_avg_sq": v[k]}
        return {"epoch": epoch, "name": name, "state_dict": sd, "optimizer": opt.state_dict()}

    def load_reference_checkpoint(self, ckpt: dict, model):
        """The inverse of reference_checkpoint, for a checkpoint the reference wrote (--resume, train_AT_text_only.py:351-372):
        the text-tower weights of ckpt["state_dict"] (any prefix: `module.`, `text.`), and the AdamW step and moments of the
        text parameters from ckpt["optimizer"]. `model` is the caller's open_clip module (or its DDP wrapper) the checkpoint
        was written from: its named_parameters() give the order of the optimizer's parameter ids. ckpt["scaler"] is ignored.
        Raises ValueError, changing nothing, if the groups do not fit the model, the text parameters' steps disagree, or the
        groups' lr / betas / eps / weight_decay differ from this trainer's (set trainer.lr to the checkpoint's scheduled lr
        first). The checkpoint is saved at an epoch end, so no gradients are pending: micro restarts at opt_step * accum_freq."""
        self._check_idle("load_reference_checkpoint")
        groups, text = self._reference_groups(model)
        osd = ckpt["optimizer"]
        pg = osd["param_groups"]
        sizes = [len(g["params"]) for g in pg]
        if sizes != [len(g) for g in groups]:
            raise ValueError(f"optimizer groups of {sizes} parameters, the reference's groups over this model have "
                             f"{[len(g) for g in groups]}")
        bad = []
        for i, (g, wd) in enumerate(zip(pg, (0.0, self.wd))):
            for key, want in (("lr", self.lr), ("betas", (self.beta1, self.beta2)), ("eps", self.eps), ("weight_decay", wd)):
                got = tuple(g[key]) if key == "betas" else g[key]
                if got != want:
                    bad.append(f"group {i} {key}: {got!r} in the checkpoint, {want!r} in this trainer")
        state, steps = {}, {}
        for pid, p in zip([pid for g in pg for pid in g["params"]], groups[0] + groups[1]):
            k = text.get(id(p))
            if k is not None:
                state[k] = osd["state"].get(pid)
                steps[k] = int(state[k]["step"]) if state[k] else 0
                if state[k] and tuple(state[k]["exp_avg"].shape) != tuple(p.shape):
                    bad.append(f"moments of {k}: shape {tuple(state[k]['exp_avg'].shape)}, the parameter has {tuple(p.shape)}")
        by_step = {}
        for k, s in steps.items():
            by_step.setdefault(s, []).append(k)
        if len(by_step) > 1:
            bad.append("the text parameters' AdamW steps disagree: " +
                       "; ".join(f"step {s} for {len(ks)} of them ({ks[0]}, ...)" for s, ks in by_step.items()))
        if bad:
            raise ValueError("reference checkpoint does not fit this trainer: " + "; ".join(bad))
        self.tower.load_open_clip_state_dict(ckpt["state_dict"])            # checks its keys before it copies
        step = next(iter(steps.values()))
        with torch.no_grad():
            for moment, flat in (("exp_avg", self.exp_avg), ("exp_avg_sq", self.exp_avg_sq)):
                if not step:
                    flat.zero_()
                    continue
                for k, view in self._by_name(flat).items():
                    view.copy_(state[k][moment])
        self.tower.zero_grad()
        self.opt_step, self.micro = step, step * self.accum_freq
