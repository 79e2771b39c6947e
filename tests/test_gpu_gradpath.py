"""Gradient path without a scale / pack pass: loss-seed weighting (fused CE kernel), gradient sinks (backward kernels write
into the flat symmetric buffer) and the precision modes (bf16 / tf32) of a full DenseNet step vs a plain fp32 torch model."""
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "gradpath.npz")


@pytest.fixture(scope="module")
def nat():
    from dynamic_load_balance_distributeddnn_b200.ops import _native
    assert _native.available()
    return _native


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("b,c", [(512, 10), (37, 100), (8, 1000)])
def test_fused_cross_entropy_kernel(nat, dtype, b, c):
    from dynamic_load_balance_distributeddnn_b200 import ops
    torch.manual_seed(b + c)
    x = (torch.randn(b, c, device="cuda") * 3).to(dtype).requires_grad_(True)
    y = torch.randint(0, c, (b,), device="cuda")
    scale = torch.tensor([0.375], device="cuda")
    loss = ops.cross_entropy(x, y, grad_scale=scale)
    loss.backward()
    xr = x.detach().float().requires_grad_(True)
    lr = F.cross_entropy(xr, y)
    lr.backward()
    assert abs(loss.item() - lr.item()) < 1e-4 * max(1.0, abs(lr.item()))
    tol = 1e-5 if dtype == torch.float32 else 1e-2
    assert (x.grad.float() - 0.375 * xr.grad).abs().max().item() < tol * max(1e-3, xr.grad.abs().max().item())


def _trainer(tmp_path, tag, dtype="bf16", model="densenet", bs=32, **env):
    from dynamic_load_balance_distributeddnn_b200.config import DBSConfig
    from dynamic_load_balance_distributeddnn_b200.engine import Trainer
    from dynamic_load_balance_distributeddnn_b200.utils import init_logger
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        cfg = DBSConfig(debug=False, world_size=1, batch_size=bs, model=model, dataset="cifar10", synthetic=True,
                        train_samples=bs * 8, test_samples=64, epoch_size=1, validate=False, cuda_graphs=False, dtype=dtype,
                        learning_rate=0.05, log_dir=str(tmp_path / f"l{tag}"), stats_dir=str(tmp_path / "s"))
        t = Trainer(cfg, 0, 1, "cuda:0", init_logger(cfg, 0, stream=False))
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    t.train_set.pad, t.train_set.flip = 0, False
    return t


def _run_steps(t, n, bs=32):
    for s in range(n):
        xb, yb = t.stager.stage(list(range(s * bs, s * bs + bs)))
        t.train_step(xb, yb)
        t.stager.release()
    torch.cuda.synchronize()


def test_gradient_sinks_match_pack_path(nat, tmp_path):
    """same 4 steps with the sinks on (wgrad / GN affine grads written into the flat buffer) and off (.grad + pack)"""
    a = _trainer(tmp_path, "a", DLB_GRAD_SINKS=1)
    b = _trainer(tmp_path, "b", DLB_GRAD_SINKS=0)
    assert a.flat.sinks_enabled and not b.flat.sinks_enabled and a.flat.seed_weighting
    _run_steps(a, 4); _run_steps(b, 4)
    assert not any(a.flat._sunk)
    d = (a.flat.master - b.flat.master).abs().max().item()
    moved = (a.flat.master - _trainer(tmp_path, "c").flat.master).abs().max().item()
    assert moved > 1e-3 and d < 0.05 * moved, (d, moved)
    assert a.flat.grad_in.abs().max().item() == 0.0          # cleared by the optimizer step for the next accumulation
    assert abs(a.loss_acc.item() - b.loss_acc.item()) < 2e-2 * abs(b.loss_acc.item())
    a.close(); b.close()


def gradient_sample(numels, budget=1024, seed=0):
    """Stratified sample of a model's parameters: every tensor gets a share of ``budget`` proportional to its size (at least
    one element).  Returns (tensor index, element index) arrays."""
    rng = np.random.RandomState(seed)
    total = sum(numels)
    ti, ei = [], []
    for i, n in enumerate(numels):
        k = min(n, max(1, round(budget * n / total)))
        ti.append(np.full(k, i))
        ei.append(np.sort(rng.choice(n, k, replace=False)))
    return np.concatenate(ti), np.concatenate(ei)


def _flat_sample(params, ti, ei):
    return torch.cat([p.detach().float().reshape(-1)[torch.as_tensor(ei[ti == i], device=p.device)]
                      for i, p in enumerate(params)]).cpu().numpy()


def _step_matches_reference(t, case, tol):
    """One optimisation step (augment off) of trainer ``t`` on images 0..15 vs the reference model's fp32 step on the same
    weights and images, recorded under tests/golden/ by tools/make_golden.py: the loss, and the relative L2 distance of the
    update / lr (= the gradient: first step, empty momentum buffer) from the reference gradient, estimated on a stratified
    sample of every parameter tensor."""
    gold = np.load(GOLDEN)
    pre = case + "/"
    params = [p for _, p in t.model.named_parameters()]
    numel = np.array([p.numel() for p in params])
    assert numel.tolist() == gold[pre + "numel"].tolist(), "parameter layout differs from the recorded reference model"
    ti, ei = gradient_sample(numel.tolist())
    xb, yb = t.stager.stage(list(range(16)))
    x = t._prepare_images(xb).double()
    assert yb.tolist() == gold[pre + "labels"].tolist()
    assert abs(x.sum().item() - float(gold[pre + "x_sum"])) < 1e-4 * x.abs().sum().item(), "inputs differ from the recording"
    before = _flat_sample(params, ti, ei)
    np.testing.assert_allclose(before, gold[pre + "w0"], rtol=1e-6, atol=1e-7, err_msg="initial weights differ from the recording")
    t.train_step(xb, yb)
    t.stager.release()
    torch.cuda.synchronize()
    loss_ref = float(gold[pre + "loss"])
    assert abs(t.loss_acc.item() - loss_ref) < tol * max(1.0, loss_ref), (t.loss_acc.item(), loss_ref)
    upd = (before - _flat_sample(params, ti, ei)) / 0.05
    g = gold[pre + "grad"]
    w = (numel / np.bincount(ti, minlength=len(numel)))[ti]       # stratum weight of each sampled element
    rel = math.sqrt(float((w * (upd - g) ** 2).sum() / (w * g ** 2).sum()))
    assert rel < 3 * tol, rel


@pytest.mark.parametrize("dtype,tol", [("tf32", 2e-2), ("bf16", 0.15)])
def test_densenet_step_matches_fp32_torch_model(nat, tmp_path, dtype, tol):
    """one full optimisation step (augment off) of the native DenseNet-121 vs the same step of the reference's own
    DenseNet-121 (stock torch.nn layers, fp32) on the same weights: loss and parameter update."""
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    t = _trainer(tmp_path, dtype, dtype=dtype, bs=16)
    _step_matches_reference(t, "densenet-" + dtype, tol)
    t.close()


def test_tf32_training_decreases_loss_like_bf16(nat, tmp_path):
    """convergence parity on the synthetic learnable set: tf32 and bf16 runs of the same 40 steps end at similar losses"""
    finals = {}
    for dtype in ("tf32", "bf16"):
        t = _trainer(tmp_path, "conv" + dtype, dtype=dtype, model="resnet18", bs=64)
        losses = []
        for s in range(40):
            xb, yb = t.stager.stage(list(range((s % 8) * 64, (s % 8) * 64 + 64)))
            t.loss_acc.zero_()
            t.train_step(xb, yb)
            t.stager.release()
            losses.append(t.loss_acc.item())
        finals[dtype] = (sum(losses[:5]) / 5, sum(losses[-5:]) / 5)
        t.close()
    for dtype, (first, last) in finals.items():
        assert last < 0.8 * first, (dtype, first, last)
    assert abs(finals["tf32"][1] - finals["bf16"][1]) < 0.25 * finals["tf32"][0], finals


@pytest.mark.parametrize("model,ref_mod,ref_cls,dtype,tol", [
    ("resnet18", "Resnet", "ResNet18", "bf16", 0.15), ("resnet50", "Resnet", "ResNet50", "bf16", 0.15),
    ("regnet", "RegNet", "RegNetY_400MF", "bf16", 0.2), ("resnet18", "Resnet", "ResNet18", "tf32", 3e-2),
    ("regnet", "RegNet", "RegNetY_400MF", "tf32", 3e-2)])
def test_family_step_matches_reference_model(nat, tmp_path, model, ref_mod, ref_cls, dtype, tol):
    """Full optimisation step of a zoo family through the native kernels (GN fusions, tcgen05 convs, SE / stem kernels, flat
    optimizer) vs the REFERENCE's own class ``ref_mod.ref_cls`` (stock torch.nn, true fp32) on the same weights: loss +
    relative L2 of the update."""
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    t = _trainer(tmp_path, model + dtype, dtype=dtype, model=model, bs=16)
    _step_matches_reference(t, f"{model}-{dtype}", tol)
    t.close()
