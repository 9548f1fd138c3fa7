"""Fused Adam / AdamW over ONE flat fp32 buffer (reference src/train.py:127-128,227-233).

`FusedAdam(model.parameters(), lr=1e-4)` has torch.optim.Adam's semantics (dense grads,
betas=(0.9,0.999), eps=1e-8).  On construction the parameters are re-pointed into one flat
device buffer and their `.grad` into one flat gradient buffer, so that
  * the update is a single libnrms_b200 launch streaming 4 reads + 3 writes per element, and
  * data-parallel training needs exactly one NCCL all-reduce per step (`allreduce_grads`).
Parameter names/shapes (state_dict) are untouched; `load_state_dict` copies in place.  `step()` bumps every parameter's
version counter, as an in-place torch op would.
"""
from __future__ import annotations

import math

import torch

from . import ops


class FusedAdam(torch.optim.Optimizer):
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, decoupled=False):
        defaults = dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, decoupled=decoupled)
        super().__init__(params, defaults)
        if len(self.param_groups) != 1:
            raise ValueError("FusedAdam keeps one flat buffer: pass a single parameter group")
        ps = [p for p in self.param_groups[0]["params"] if p.requires_grad]
        if not ps:
            raise ValueError("no trainable parameters")
        dev = ps[0].device
        if dev.type != "cuda":
            raise RuntimeError("FusedAdam needs CUDA parameters (move the model first, like src/train.py:106)")
        offs, total = [], 0
        for p in ps:
            offs.append(total)
            total += (p.numel() + 3) // 4 * 4          # keep every view 16-byte aligned
        self.flat_param = torch.zeros(total, dtype=torch.float32, device=dev)
        self.flat_grad = torch.zeros(total, dtype=torch.float32, device=dev)
        self.exp_avg = torch.zeros(total, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(total, dtype=torch.float32, device=dev)
        with torch.no_grad():
            for p, o in zip(ps, offs):
                view = self.flat_param[o:o + p.numel()].view_as(p)
                view.copy_(p.data)
                p.data = view
                p.grad = self.flat_grad[o:o + p.numel()].view_as(p)
                p._nrms_grad_sink = True   # its .grad is a live view of flat_grad: the news encoder may scatter into it
        self._params, self._offsets = ps, offs
        self.step_count = 0
        # data parallel: every replica starts from rank 0's parameters (the gradient all-reduce keeps them identical from
        # then on; replicas built from different seeds would otherwise diverge silently)
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.broadcast(self.flat_param, src=0)

    def zero_grad(self, set_to_none=False):
        # keep the .grad views alive (autograd accumulates into them in place)
        self.flat_grad.zero_()
        for p, o in zip(self._params, self._offsets):
            if p.grad is None or p.grad.data_ptr() != self.flat_grad.data_ptr() + 4 * o:
                p.grad = self.flat_grad[o:o + p.numel()].view_as(p)

    def allreduce_grads(self):
        """One collective over the flat gradient; returns the scale step() must apply (1/world)."""
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(self.flat_grad)
            return 1.0 / dist.get_world_size()
        return 1.0

    @torch.no_grad()
    def step(self, closure=None, grad_scale=1.0):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        g = self.param_groups[0]
        for p, o in zip(self._params, self._offsets):     # a grad that autograd re-allocated is folded back in
            if p.grad is not None and p.grad.data_ptr() != self.flat_grad.data_ptr() + 4 * o:
                self.flat_grad[o:o + p.numel()].view_as(p).add_(p.grad)
                p.grad = self.flat_grad[o:o + p.numel()].view_as(p)
        self.step_count += 1
        ops.adam_step_(self.flat_param, self.flat_grad, self.exp_avg, self.exp_avg_sq, self.step_count,
                       lr=g["lr"], betas=g["betas"], eps=g["eps"], weight_decay=g["weight_decay"],
                       decoupled=g["decoupled"], grad_scale=grad_scale)
        # the kernel writes through raw pointers, which autograd does not see: bump every parameter's version counter so
        # caches keyed on it (MultiHeadSelfAttention.packed, Recommender) rebuild and saved-tensor checks hold
        torch.autograd.graph.increment_version(self._params)
        return loss


    # ---- checkpoint interchange with torch.optim.Adam / AdamW (reference src/train.py:266-277 saves
    #      optimizer.state_dict() next to model.state_dict()) ------------------------------------------------
    def state_dict(self):
        """torch.optim.Adam's layout: per-parameter `step` / `exp_avg` / `exp_avg_sq` (clones, not views of the flat
        buffers) and one param group, so a reference checkpoint written from this optimizer loads into
        torch.optim.Adam(model.parameters()) and vice versa."""
        g = self.param_groups[0]
        state = {}
        if self.step_count > 0:
            for i, (p, o) in enumerate(zip(self._params, self._offsets)):
                state[i] = dict(step=torch.tensor(float(self.step_count)),
                                exp_avg=self.exp_avg[o:o + p.numel()].view_as(p).clone(),
                                exp_avg_sq=self.exp_avg_sq[o:o + p.numel()].view_as(p).clone())
        group = dict(lr=g["lr"], betas=tuple(g["betas"]), eps=g["eps"], weight_decay=g["weight_decay"], amsgrad=False,
                     maximize=False, foreach=None, capturable=False, differentiable=False, fused=None,
                     decoupled_weight_decay=bool(g["decoupled"]), params=list(range(len(self._params))))
        return dict(state=state, param_groups=[group])

    @torch.no_grad()
    def load_state_dict(self, state_dict):
        groups = state_dict["param_groups"]
        if len(groups) != 1 or len(groups[0]["params"]) != len(self._params):
            raise ValueError("optimizer state has a different parameter list (expected one group of "
                             f"{len(self._params)} parameters)")
        src = groups[0]
        if src.get("amsgrad") or src.get("maximize"):
            raise ValueError("amsgrad / maximize optimizer states are not supported by the fused Adam kernel")
        g = self.param_groups[0]
        g["lr"], g["betas"], g["eps"] = src["lr"], tuple(src["betas"]), src["eps"]
        g["weight_decay"] = src.get("weight_decay", g["weight_decay"])
        if "decoupled_weight_decay" in src:
            g["decoupled"] = bool(src["decoupled_weight_decay"])
        state = state_dict["state"]
        self.exp_avg.zero_()
        self.exp_avg_sq.zero_()
        steps = set()
        for i, (p, o) in enumerate(zip(self._params, self._offsets)):
            st = state.get(src["params"][i])
            if st is None:
                continue
            if tuple(st["exp_avg"].shape) != tuple(p.shape):
                raise ValueError(f"optimizer state {i}: shape {tuple(st['exp_avg'].shape)} != parameter {tuple(p.shape)}")
            self.exp_avg[o:o + p.numel()].view_as(p).copy_(st["exp_avg"])
            self.exp_avg_sq[o:o + p.numel()].view_as(p).copy_(st["exp_avg_sq"])
            steps.add(int(float(st["step"])))
        if len(steps) > 1:
            raise ValueError(f"per-parameter step counts differ ({sorted(steps)}): one bias correction per flat buffer")
        self.step_count = steps.pop() if steps else 0


class FusedAdamW(FusedAdam):
    """torch.optim.AdamW semantics (decoupled weight decay, default 0.01)."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01):
        super().__init__(params, lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, decoupled=True)


def cosine_lr(base_lr, step, total_steps, eta_min=0.0):
    """CosineAnnealingLR closed form (config-5 variant; builder-defined, see DESIGN.md)."""
    return eta_min + (base_lr - eta_min) * (1 + math.cos(math.pi * step / total_steps)) / 2
