"""nn.SyncBatchNorm on the kernel path (unet/syncbn.py): a model converted with
``nn.SyncBatchNorm.convert_sync_batchnorm`` normalises with the statistics of every rank of its group, in bf16 and
tf32 modes, forward and backward, exactly where torch's SyncBatchNorm would, and nowhere else.

1. One process, no process group: the converted model IS the unconverted one, bit for bit, with no collective.
2. Two processes on one GPU over gloo (CUDA tensors), eager: 2 ranks x 2 images through BatchShardedTrainer equal
   one process x the same 4 images with plain BatchNorm (loss, logits, running buffers, every gradient after the
   trainer's all-reduce), 3 + 1 images give the batch-4 statistics, and the unconverted model misses by far more.
3. Two GPUs over NCCL: graph replay of the trainer equals eager, ranks stay bit-identical without buffer syncing,
   and the result matches the single-GPU batch-4 run.
"""
import copy
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn as nn

from oracle import unet_oracle as O

pytestmark = pytest.mark.gpu

H = W = 64
# rel-L2 gates of the two-rank runs against the single-process batch-4 run, about 3x (bf16) and 10x (tf32) what was
# measured on a B200.  Synchronised statistics differ from the batch-4 ones only in the order the fp64 sums are
# folded; the gradients also in the order the per-rank weight-gradient tiles are summed, and in bf16 mode in the bf16
# roundings this moves.  Measured, synchronised / per-rank: tf32 0 / 3.5e-1 (logits), 0 / 7.7e-1 (buffers),
# <= 2.3e-6 / >= 1.5e-1 (gradients); bf16 4.8e-4 / 4.0e-3 (logits), 7.0e-6 / 7.7e-1 (buffers), gradients
# 5.6e-5 / 4.7e-4 (conv weights), 2.1e-3 / 3.8e-2 (gammas), 1.3e-5 / 7.8e-5 (betas), 3.0e-3 / 5.6e-2 (psi weight).
# With every ReLU active (bf16) the per-rank statistics move logits and gradients little; the running buffers tell
# them apart by far.  The bf16 loss does not tell them apart at all (1.5e-5 per-rank) and is gated only.
GATE = {"tf32": dict.fromkeys(("loss", "logits", "buffers", "grad_conv_weight", "grad_weight", "grad_bias",
                               "grad_psi_weight"), 2e-5),
        "bf16": {"loss": 6e-5, "logits": 1.5e-3, "buffers": 3e-5, "grad_conv_weight": 2e-4, "grad_weight": 6e-3,
                 "grad_bias": 4e-5, "grad_psi_weight": 1e-2}}


def _rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def _set_precision(p):
    import unet
    unet.set_precision(p)


def _model(kind, precision, seed=5):
    from unet.models import AttentionUNet, UNet
    torch.manual_seed(seed)
    model = AttentionUNet(1, 2, True, 16) if kind == "attention" else UNet(1, 2, True, 16)
    if precision == "bf16":
        # every BatchNorm bias +8 (not psi's), so that no ReLU sits near a decision that the bf16 roundings of two
        # correct implementations take differently (as in test_channels_gpu.py)
        with torch.no_grad():
            for name, mod in model.named_modules():
                if isinstance(mod, nn.BatchNorm2d) and ".psi." not in name:
                    mod.bias.fill_(8.0)
    return model


def _data(n=4, seed=21):
    x, _ = O.synthetic_batch(n, H, W, seed=seed)
    t = torch.randint(0, 2, (n, H, W), generator=torch.Generator().manual_seed(seed))
    return x, t


class _Count:
    """torch.distributed.all_reduce with a call counter."""

    def __init__(self, monkeypatch=None):
        self.calls = 0
        self.fn = dist.all_reduce
        if monkeypatch is not None:
            monkeypatch.setattr(dist, "all_reduce", self)

    def __call__(self, *a, **k):
        self.calls += 1
        return self.fn(*a, **k)


def _bn_buffers(model):
    return [b.detach().clone() for n, b in model.named_buffers()]


# --------------------------------------------------------------------------- 1. one process
@pytest.mark.parametrize("precision", ["bf16", "tf32"])
@pytest.mark.parametrize("kind", ["attention", "unet"])
def test_single_process_converted_is_unconverted(kind, precision, monkeypatch):
    count = _Count(monkeypatch)
    _set_precision(precision)
    try:
        plain = _model(kind, precision).cuda()
        conv = nn.SyncBatchNorm.convert_sync_batchnorm(copy.deepcopy(plain))
        assert any(isinstance(m, nn.SyncBatchNorm) for m in conv.modules())
        x, _ = _data(2)
        results = []
        for model in (plain, conv):
            out = {}
            model.train()
            xi = x.cuda().requires_grad_(True)
            y = model(xi)
            (y * torch.linspace(-1, 1, y.numel(), device="cuda").view_as(y)).sum().backward()
            out["train"] = [y.detach(), xi.grad] + [p.grad.clone() for p in model.parameters()] + _bn_buffers(model)
            model.eval()
            xi = x.cuda().requires_grad_(True)
            y = model(xi)          # frozen statistics with gradients
            y.sum().backward()
            out["frozen"] = [y.detach(), xi.grad]
            with torch.no_grad():
                out["eval"] = [model(x.cuda())]
            results.append(out)
        for key in ("train", "frozen", "eval"):
            for a, b in zip(results[0][key], results[1][key]):
                assert torch.equal(a, b), key
    finally:
        _set_precision("bf16")
    assert count.calls == 0


# --------------------------------------------------------------------------- 2. two processes, gloo, one GPU
def _trainer_step(model, x, t):
    """One BatchShardedTrainer step with lr 0: returns (loss, logits of a train-mode forward before the step,
    gradients after the trainer's all-reduce).  Both forwards advance the running buffers."""
    from unet.parallel import BatchShardedTrainer
    tr = BatchShardedTrainer(model, nn.CrossEntropyLoss(), torch.optim.SGD(model.parameters(), lr=0.0),
                             buffer_sync="none")
    model.train()
    with torch.no_grad():
        logits = model(x.cuda())
    loss = tr.step(x, t)
    return loss.detach().clone(), logits, {n: p.grad.detach().clone() for n, p in model.named_parameters()}


def _gloo_worker(rank, world, root, precision):
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", init_method=f"file://{root}/init", rank=rank, world_size=world)
    try:
        _set_precision(precision)
        x, t = _data(4)
        res = {}
        for name, convert, lo, hi in (("sync", True, 2 * rank, 2 * rank + 2), ("plain", False, 2 * rank, 2 * rank + 2),
                                      ("uneven", True, (0, 3)[rank], (3, 4)[rank])):
            model = _model("attention", precision).cuda()
            if convert:
                model = nn.SyncBatchNorm.convert_sync_batchnorm(model)
            loss, logits, grads = _trainer_step(model, x[lo:hi], t[lo:hi])
            res[name] = {"loss": loss.cpu(), "logits": logits.cpu(), "grads": {k: g.cpu() for k, g in grads.items()},
                         "buffers": [b.cpu() for b in _bn_buffers(model)]}
            if name == "sync":
                count = _Count()
                dist.all_reduce = count
                try:
                    model.eval()
                    with torch.no_grad():
                        model(x[lo:hi].cuda())
                    xi = x[lo:hi].cuda().requires_grad_(True)
                    model(xi).sum().backward()
                finally:
                    dist.all_reduce = count.fn
                res["eval_collectives"] = count.calls
        torch.save(res, f"{root}/r{rank}.pt")
    finally:
        dist.destroy_process_group()


def _reference(precision, n_images=4):
    _set_precision(precision)
    try:
        x, t = _data(4)
        model = _model("attention", precision).cuda()
        loss, logits, grads = _trainer_step(model, x[:n_images], t[:n_images])
        return {"loss": loss.cpu(), "logits": logits.cpu(), "grads": {k: g.cpu() for k, g in grads.items()},
                "buffers": [b.cpu() for b in _bn_buffers(model)]}
    finally:
        _set_precision("bf16")


def _grad_group(name, g):
    """Gradients are compared per kind: with every ReLU active the BatchNorm biases of a layer that feeds another
    BatchNorm have a gradient of pure rounding noise (the next mean subtraction removes a constant shift), so one
    parameter's relative error says nothing; a kind's concatenated gradient does.  Double-counted dgamma / dbeta /
    dw_psi show up as an error of 1 in their kind."""
    if ".psi.0." in name:
        return "psi_weight"
    return "conv_weight" if g.dim() == 4 else name.rsplit(".", 1)[1]


def _grad_errors(got, ref):
    groups = {}
    for name, g in ref.items():
        groups.setdefault(_grad_group(name, g), []).append(name)
    return {k: _rel(torch.cat([got[n].flatten() for n in names]), torch.cat([ref[n].flatten() for n in names]))
            for k, names in groups.items()}


def _errors(ranks, ref, key):
    """rel-L2 of the two ranks' results (sync or plain, equal shards) against the batch-4 reference."""
    r0, r1 = ranks[0][key], ranks[1][key]
    err = {"loss": _rel((r0["loss"] + r1["loss"]) / 2, ref["loss"]),
           "logits": _rel(torch.cat([r0["logits"], r1["logits"]]), ref["logits"])}
    err["buffers"] = max(_rel(a, b) for a, b in zip(r0["buffers"], ref["buffers"]) if b.is_floating_point())
    err.update(("grad_" + k, e) for k, e in _grad_errors(r0["grads"], ref["grads"]).items())
    return err


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
def test_two_ranks_gloo_match_batch_four(precision, tmp_path):
    mp.spawn(_gloo_worker, args=(2, str(tmp_path), precision), nprocs=2, join=True)
    ranks = [torch.load(tmp_path / f"r{r}.pt", weights_only=False) for r in range(2)]
    ref = _reference(precision)
    gate = GATE[precision]
    sync, plain = _errors(ranks, ref, "sync"), _errors(ranks, ref, "plain")
    print(f"syncbn {precision}: synchronised {sync}, per-rank {plain}")
    assert set(sync) == set(gate)
    for k, e in sync.items():
        assert e <= gate[k], (k, e)
    # per-rank statistics must miss: by far in the buffers, and in tf32 everywhere
    assert plain["buffers"] > 1000 * gate["buffers"], plain
    far = 20 if precision == "tf32" else 1
    assert all(plain[k] > far * gate[k] for k in plain if k != "loss" or precision == "tf32"), plain
    for a, b in zip(ranks[0]["sync"]["buffers"], ranks[1]["sync"]["buffers"]):
        assert torch.equal(a, b)                # every rank holds the global running statistics
    for k in ranks[0]["sync"]["grads"]:
        assert torch.equal(ranks[0]["sync"]["grads"][k], ranks[1]["sync"]["grads"][k]), k
    assert ranks[0]["eval_collectives"] == 0 and ranks[1]["eval_collectives"] == 0
    # 3 + 1 images: the batch-4 statistics (running buffers) and logits
    uneven = ranks[0]["uneven"], ranks[1]["uneven"]
    assert _rel(torch.cat([uneven[0]["logits"], uneven[1]["logits"]]), ref["logits"]) <= gate["logits"]
    for a, b, c in zip(uneven[0]["buffers"], uneven[1]["buffers"], ref["buffers"]):
        assert torch.equal(a, b)
        if c.is_floating_point():
            assert _rel(a, c) <= gate["buffers"]
        else:
            assert torch.equal(a, c)


# --------------------------------------------------------------------------- 3. two GPUs, NCCL, graph replay
STEPS = 4


def _nccl_worker(rank, world, root, precision):
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"file://{root}/init", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    try:
        from unet.optim import FusedAdamW
        from unet.parallel import BatchShardedTrainer
        _set_precision(precision)
        x, t = _data(4)
        res = {}
        for use_graph in (False, True):
            model = nn.SyncBatchNorm.convert_sync_batchnorm(_model("attention", precision)).cuda()
            tr = BatchShardedTrainer(model, nn.CrossEntropyLoss(), FusedAdamW(model.parameters(), lr=1e-4),
                                     grad_clip=1.0, cuda_graph=use_graph, graph_warmup=2, buffer_sync="none")
            losses = [tr.step(x[2 * rank:2 * rank + 2], t[2 * rank:2 * rank + 2]) for _ in range(STEPS)]
            torch.cuda.synchronize()
            res[use_graph] = {"losses": torch.stack(losses).cpu(),
                              "params": [p.detach().cpu() for p in model.parameters()],
                              "buffers": [b.cpu() for b in _bn_buffers(model)]}
            tr.release_graphs()
        torch.save(res, f"{root}/r{rank}.pt")
    finally:
        dist.destroy_process_group()


def _nccl_reference(precision):
    from unet.optim import FusedAdamW
    from unet.parallel import BatchShardedTrainer
    _set_precision(precision)
    try:
        x, t = _data(4)
        model = _model("attention", precision).cuda()
        tr = BatchShardedTrainer(model, nn.CrossEntropyLoss(), FusedAdamW(model.parameters(), lr=1e-4), grad_clip=1.0)
        losses = [tr.step(x, t) for _ in range(STEPS)]
        return {"losses": torch.stack(losses).cpu(), "params": [p.detach().cpu() for p in model.parameters()],
                "buffers": [b.cpu() for b in _bn_buffers(model)]}
    finally:
        _set_precision("bf16")


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("precision", ["tf32", "bf16"])
def test_two_gpus_nccl_graph_replay(precision, tmp_path):
    mp.spawn(_nccl_worker, args=(2, str(tmp_path), precision), nprocs=2, join=True)
    ranks = [torch.load(tmp_path / f"r{r}.pt", weights_only=False) for r in range(2)]
    for r in ranks:
        for key in ("losses", "params", "buffers"):
            a, b = r[False][key], r[True][key]
            for u, v in zip(a if isinstance(a, list) else [a], b if isinstance(b, list) else [b]):
                assert torch.equal(u, v), key           # replay == eager
    for key in ("params", "buffers"):
        for u, v in zip(ranks[0][True][key], ranks[1][True][key]):
            assert torch.equal(u, v), key               # replicas bit-identical with buffer_sync="none"
    ref = _nccl_reference(precision)
    gate = GATE[precision]["logits"]
    assert _rel((ranks[0][True]["losses"] + ranks[1][True]["losses"]) / 2, ref["losses"]) <= gate
    assert max(_rel(a, b) for a, b in zip(ranks[0][True]["params"], ref["params"])) <= gate
    assert max(_rel(a, b) for a, b in zip(ranks[0][True]["buffers"], ref["buffers"])
               if b.is_floating_point()) <= gate
