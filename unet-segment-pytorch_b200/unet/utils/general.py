"""``ModelEMA`` — drop-in for ``unet.utils.general.ModelEMA`` of the reference
(unet/utils/general.py:111-199), with ``update()`` as ONE multi-tensor CUDA launch.

The reference's update walks ``named_parameters()`` / ``named_buffers()`` and issues two small
kernels per parameter and one per buffer (~250 launches per step for an AttentionUNet, more host
time than a whole batch-4 training step on a B200).  Same constructor, attributes (``ema_model``,
``decay``, ``warmup_steps``, ``updates``), ``update`` / ``state_dict`` / ``load_state_dict``; the
decay lives in device memory so the update can be captured into the trainer's step graph.
"""
from __future__ import annotations

import copy

import torch

from .. import _C
from .. import kernels as K


class ModelEMA:
    def __init__(self, model: torch.nn.Module, decay: float = 0.999, warmup_steps: int = 0):
        self.decay = decay
        self.warmup_steps = warmup_steps
        self.updates = 0
        self.ema_model = copy.deepcopy(model)
        self.ema_model.eval()
        for param in self.ema_model.parameters():
            param.requires_grad_(False)
        self._tables = None   # (signature, desc, chunks, nchunks, decay tensor)
        self._decay_host = None

    # ------------------------------------------------------------------ tables
    def _pairs(self, model):
        src_p, src_b = dict(model.named_parameters()), dict(model.named_buffers())
        pairs = []
        for name, e in self.ema_model.named_parameters():
            if name in src_p:
                pairs.append((e, src_p[name], 0))
        for name, e in self.ema_model.named_buffers():
            if name in src_b:
                pairs.append((e, src_b[name], 2 if e.dtype == torch.int64 else 1))
        return pairs

    def _build(self, model):
        pairs = self._pairs(model)
        for e, s, kind in pairs:
            ok = (e.is_cuda and s.is_cuda and e.is_contiguous() and s.is_contiguous() and e.dtype == s.dtype
                  and e.numel() == s.numel() and e.dtype in (torch.float32, torch.int64))
            if not ok:
                raise RuntimeError("ModelEMA needs contiguous fp32 (int64 counters) CUDA parameters and buffers "
                                   "(no CPU fallback)")
        dev = pairs[0][0].device
        ce = int(_C.lib().ub2_adamw_chunk_elems())
        desc = [[e.data_ptr(), s.data_ptr(), e.numel(), kind] for e, s, kind in pairs]
        chunks = [(t, off) for t, (e, _, _) in enumerate(pairs) for off in range(0, e.numel(), ce)]
        sig = tuple(d[0] for d in desc) + tuple(d[1] for d in desc)
        self._tables = (sig, torch.tensor(desc, dtype=torch.int64).to(dev),
                        torch.tensor(chunks, dtype=torch.int32).to(dev), len(chunks),
                        torch.zeros(1, device=dev, dtype=torch.float32))
        self._decay_host = None

    def _signature(self, model):
        pairs = self._pairs(model)
        return tuple(e.data_ptr() for e, _, _ in pairs) + tuple(s.data_ptr() for _, s, _ in pairs)

    def _current_decay(self) -> float:
        if self.updates <= self.warmup_steps:
            return min(self.decay, (1 + self.updates) / (10 + self.updates))
        return self.decay

    def prepare(self, model: torch.nn.Module) -> None:
        """Host side of one update: (re)build the pointer tables if a tensor moved, advance the
        counter and put this step's decay into device memory.  The trainer calls it before
        replaying a captured step that contains ``update(model, _advance=False)``."""
        if self._tables is None or self._tables[0] != self._signature(model):
            self._build(model)
        self.updates += 1
        d = float(self._current_decay())
        if d != self._decay_host:
            self._tables[4].fill_(d)
            self._decay_host = d

    # ------------------------------------------------------------------ reference API
    @torch.no_grad()
    def update(self, model: torch.nn.Module, _advance: bool = True) -> None:
        if _advance:
            self.prepare(model)
        elif self._tables is None:
            raise RuntimeError("ModelEMA: call prepare(model) before update(model, _advance=False)")
        _, desc, chunks, nchunks, decay = self._tables
        K.ema_update(desc, chunks, nchunks, decay)

    def state_dict(self) -> dict:
        return {'ema_state_dict': self.ema_model.state_dict(), 'decay': self.decay, 'updates': self.updates}

    def load_state_dict(self, state_dict: dict) -> None:
        self.ema_model.load_state_dict(state_dict['ema_state_dict'])
        self.decay = state_dict.get('decay', self.decay)
        self.updates = state_dict.get('updates', 0)


# set_seed, get_device, load_config, increment_path (general.py:18-108 of the reference) are host-side
# orchestration: they resolve to the attached reference checkout's own general.py (unet/overlay.py)
from .. import overlay as _overlay  # noqa: E402

__getattr__ = _overlay.module_getattr(__name__, "utils/general.py")
