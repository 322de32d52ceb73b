"""Fused optimizer tail: gradient-norm clipping + AdamW in two multi-tensor CUDA launches.

The reference's step is ``clip_grad_norm_(model.parameters(), grad_clip)`` (scripts/train.py:141)
followed by ``torch.optim.AdamW(...).step()`` (built at scripts/train.py:346-350).  ``FusedAdamW``
takes the same constructor arguments as ``torch.optim.AdamW``, keeps its ``state_dict`` format
(``step`` / ``exp_avg`` / ``exp_avg_sq`` per parameter, so checkpoints written by either load
into the other) and runs the same arithmetic through ``ub2_grad_sumsq`` + ``ub2_adamw_step``
(csrc/optim.cu).  Step count and hyper-parameters live in device memory: the step is
CUDA-graph capturable and a learning-rate scheduler keeps working under graph replay
(``sync_hyperparams()`` copies the current values in, outside the graph).
"""
from __future__ import annotations

import torch

from . import _C
from . import kernels as K


class FusedAdamW(torch.optim.AdamW):
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, amsgrad=False,
                 *, max_grad_norm: float = 0.0, write_clipped_grads: bool = False, **kwargs):
        if amsgrad:
            raise NotImplementedError("FusedAdamW: amsgrad is not supported")
        if kwargs.pop("maximize", False):
            raise NotImplementedError("FusedAdamW: maximize is not supported")
        for k in ("foreach", "capturable", "fused", "differentiable"):
            kwargs.pop(k, None)
        super().__init__(params, lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, amsgrad=False)
        self.max_grad_norm = float(max_grad_norm)
        self.write_clipped_grads = bool(write_clipped_grads)
        self._fz = None  # lazily built flat state + device tables

    # ------------------------------------------------------------------ state plumbing
    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        self._fz = None   # re-flatten the loaded moments on the next step

    def zero_grad(self, set_to_none: bool = False):
        """Zero the gradients IN PLACE by default (torch's default drops them): the flat state and the
        device pointer tables are keyed on the gradient buffers, and a loop in the reference's style
        (``optimizer.zero_grad()`` after every step, train.py:143) would otherwise re-allocate every
        gradient and make each step rebuild them.  ``set_to_none=True`` still works, at that price."""
        if set_to_none:
            return super().zero_grad(set_to_none=True)
        for g in self.param_groups:
            grads = [p.grad for p in g["params"] if p.grad is not None]
            if grads:
                torch._foreach_zero_(grads)

    def add_param_group(self, param_group):
        super().add_param_group(param_group)
        self._fz = None

    def state_dict(self):
        """torch.optim.AdamW's format: per-parameter ``step`` as a CPU float tensor."""
        if self._fz is not None:
            step_cpu = self._fz["step"].detach().cpu().reshape(())
            for p in self._fz["params"]:
                self.state[p]["step"] = step_cpu.clone()
        sd = super().state_dict()
        sd["state"] = {k: dict(v) for k, v in sd["state"].items()}   # detach from the live state dicts
        if self._fz is not None:
            for p in self._fz["params"]:
                self.state[p]["step"] = self._fz["step"][0]
        return sd

    def _hyper_rows(self):
        rows = []
        for gi, g in enumerate(self.param_groups):
            lr = g["lr"]
            lr = float(lr.item()) if isinstance(lr, torch.Tensor) else float(lr)
            b1, b2 = g["betas"]
            rows.append([lr, float(b1), float(b2), float(g["eps"]), float(g["weight_decay"]),
                         self.max_grad_norm if gi == 0 else 0.0, 0.0, 0.0])
        return rows

    def _build(self):
        params, groups = [], []
        for gi, g in enumerate(self.param_groups):
            for p in g["params"]:
                if p.grad is None:
                    continue
                if not (p.is_cuda and p.dtype == torch.float32 and p.is_contiguous()
                        and p.grad.dtype == torch.float32 and p.grad.is_contiguous()):
                    raise RuntimeError("FusedAdamW needs contiguous fp32 CUDA parameters and gradients "
                                       "(no CPU fallback)")
                params.append(p)
                groups.append(gi)
        if not params:
            raise RuntimeError("FusedAdamW.step(): no parameter has a gradient")
        dev = params[0].device
        pad = lambda n: (n + 3) & ~3
        total = sum(pad(p.numel()) for p in params)
        flat_m = torch.zeros(total, device=dev, dtype=torch.float32)
        flat_v = torch.zeros(total, device=dev, dtype=torch.float32)
        step = torch.zeros(1, device=dev, dtype=torch.float32)
        loaded_steps = []
        off = 0
        ptrs = [[], [], [], []]
        for p in params:
            n = p.numel()
            m = flat_m[off:off + n].view_as(p)
            v = flat_v[off:off + n].view_as(p)
            st = self.state[p]
            if "exp_avg" in st:           # state loaded from a checkpoint (or built by torch's AdamW)
                m.copy_(st["exp_avg"])
                v.copy_(st["exp_avg_sq"])
                loaded_steps.append(st.get("step", 0))
            st["exp_avg"], st["exp_avg_sq"], st["step"] = m, v, step[0]
            ptrs[0].append(p.data_ptr()); ptrs[1].append(p.grad.data_ptr())
            ptrs[2].append(m.data_ptr()); ptrs[3].append(v.data_ptr())
            off += pad(n)
        if loaded_steps:
            # one shared step counter: read the loaded values with ONE host sync and refuse a state whose
            # parameters disagree (a param group added later, a hand-edited checkpoint) instead of
            # silently letting the last one win
            dev_steps = [s.detach().float().reshape(()) for s in loaded_steps if isinstance(s, torch.Tensor) and s.is_cuda]
            vals = [float(s) for s in loaded_steps if not (isinstance(s, torch.Tensor) and s.is_cuda)]
            if dev_steps:
                vals += torch.stack(dev_steps).cpu().tolist()
            if len(loaded_steps) != len(params) and max(vals) > 0:
                raise RuntimeError("FusedAdamW keeps one step counter for all parameters: the loaded state has "
                                   "moments for only some of them")
            if max(vals) != min(vals):
                raise RuntimeError(f"FusedAdamW keeps one step counter for all parameters: the loaded state has "
                                   f"steps from {min(vals):g} to {max(vals):g}")
            step.fill_(vals[0])
        ce = int(_C.lib().ub2_adamw_chunk_elems())
        chunks = [(t, s) for t, p in enumerate(params) for s in range(0, p.numel(), ce)]
        i64 = lambda x: torch.tensor(x, dtype=torch.int64).to(dev)
        self._fz = {
            "params": params, "step": step, "flat_m": flat_m, "flat_v": flat_v,
            "ptrs": i64(ptrs), "numel": i64([p.numel() for p in params]),
            "group": torch.tensor(groups, dtype=torch.int32).to(dev),
            "chunks": torch.tensor(chunks, dtype=torch.int32).to(dev), "nchunks": len(chunks),
            "partial": torch.empty(len(chunks), device=dev, dtype=torch.float64),
            "hyper": torch.zeros((len(self.param_groups), 8), device=dev, dtype=torch.float32),
            "hyper_host": None, "total_norm": torch.zeros(1, device=dev, dtype=torch.float32),
            "sig": tuple(ptrs[0]) + tuple(ptrs[1]),
        }
        self.sync_hyperparams()

    def sync_hyperparams(self):
        """Copy lr / betas / eps / weight decay / max norm to the device if they changed.  Call
        before replaying a captured step (the captured kernels read them from device memory)."""
        fz = self._fz
        if fz is None:
            return
        rows = self._hyper_rows()
        if rows != fz["hyper_host"]:
            fz["hyper"].copy_(torch.tensor(rows, dtype=torch.float32), non_blocking=False)
            fz["hyper_host"] = rows

    def _signature(self):
        ps, gs = [], []
        for g in self.param_groups:
            for p in g["params"]:
                if p.grad is not None:
                    ps.append(p.data_ptr())
                    gs.append(p.grad.data_ptr())
        return tuple(ps) + tuple(gs)

    # ------------------------------------------------------------------ the step
    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        capturing = torch.cuda.is_current_stream_capturing()
        if not capturing:
            if self._fz is None or self._fz["sig"] != self._signature():
                self._build()
            self.sync_hyperparams()
        elif self._fz is None:
            raise RuntimeError("FusedAdamW: run at least one eager step before capturing a CUDA graph")
        fz = self._fz
        t = len(fz["params"])
        K.grad_sumsq(fz["ptrs"], fz["numel"], fz["chunks"], fz["nchunks"], t, fz["partial"], fz["step"])
        K.adamw_step(fz["ptrs"], fz["numel"], fz["group"], fz["chunks"], fz["nchunks"], t, fz["partial"], fz["hyper"],
                     fz["step"], fz["total_norm"], self.write_clipped_grads)
        return loss

    @property
    def total_grad_norm(self) -> torch.Tensor:
        """Gradient norm measured by the last step (what clip_grad_norm_ returns), on device."""
        return self._fz["total_norm"][0] if self._fz is not None else torch.zeros(())
