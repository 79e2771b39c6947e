"""Model-zoo parity (SURVEY §2.6, §4): parameter / tensor counts, state_dict interchange and forward
equality with the reference ``Net/*`` classes.

The reference side is stored under ``tests/golden/`` (written by ``tools/make_golden.py`` from a checkout of the reference):
for each class, the key / shape / dtype of every state_dict entry and its output on a seeded input after the state was
filled with ``filled_state``.  Loading the same filled state into our model (strict) and comparing the outputs checks both
the interchange and the forward equality without the reference's sources."""
import json
import math
import os
import zlib

import numpy as np
import pytest
import torch

from dynamic_load_balance_distributeddnn_b200.models import build_model, model_names

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
EXPECTED = {"mnistnet": (21840, 8), "resnet": (42512970, 314), "resnet50": (23520842, 161),
            "densenet": (6956298, 362), "googlenet": (6166250, 258), "regnet": (5714362, 303),
            "transformer": (13828478, 27)}


@pytest.mark.parametrize("name", sorted(EXPECTED))
def test_param_counts(name):
    m = build_model(name, 10)
    ps = list(m.parameters())
    assert (sum(p.numel() for p in ps), len(ps)) == EXPECTED[name]


def test_every_registered_model_builds_and_runs():
    x = torch.randn(2, 3, 32, 32)
    for name in model_names():
        if name in ("transformer", "mnistnet") or name in ("resnet152", "densenet161", "densenet201", "resnet101", "resnet"):
            continue
        m = build_model(name, 100).eval()
        with torch.no_grad():
            assert m(x).shape == (2, 100), name


def filled_state(spec):
    """A state_dict for the entries ``spec`` = [(key, shape, dtype)], with values that depend on the key and shape only
    (weights ~ N(0, 1/fan_in), norm scales ~ 1, running variances in [0.5, 1.5)), so a model and its reference counterpart
    can be put into the same state without sharing an initialisation order."""
    sd = {}
    for key, shape, dtype in spec:
        dt = getattr(torch, dtype)
        if not dt.is_floating_point:
            sd[key] = torch.zeros(shape, dtype=dt)
            continue
        g = torch.Generator().manual_seed(zlib.crc32(key.encode()))
        if len(shape) >= 2:
            t = torch.randn(shape, generator=g) / math.sqrt(math.prod(shape[1:]))
        elif key.endswith("running_var"):
            t = 0.5 + torch.rand(shape, generator=g)
        elif key.endswith("weight"):
            t = 1.0 + 0.1 * torch.randn(shape, generator=g)
        else:
            t = 0.1 * torch.randn(shape, generator=g)
        sd[key] = t.to(dt)
    return sd


def parity_input(ctor):
    g = torch.Generator().manual_seed(0)
    if ctor == "TransformerModel":
        return torch.randint(0, 1000, (35, 3), generator=g)
    return torch.randn(2, 1, 28, 28, generator=g) if ctor == "MnistNet" else torch.randn(2, 3, 32, 32, generator=g)


def transformer_view(out):
    """The stored part of the [35, 3, 1000] log-probabilities: 16 vocabulary columns and the sum over the vocabulary."""
    return torch.cat([out[..., :16].reshape(-1), out.sum(-1).reshape(-1)])


def _golden(ctor):
    with open(os.path.join(GOLDEN, "model_parity.json")) as f:
        spec = json.load(f)[ctor]
    return [(k, tuple(shape), dt) for k, shape, dt in spec], torch.from_numpy(np.load(os.path.join(GOLDEN, "model_parity.npz"))[ctor])


@pytest.mark.parametrize("fname,ctor,ours", [("Densenet.py", "DenseNet121", "densenet"), ("Resnet.py", "ResNet50", "resnet50"),
                                              ("Resnet.py", "ResNet18", "resnet18"), ("RegNet.py", "RegNetY_400MF", "regnet"),
                                              ("MnistNet.py", "MnistNet", "mnistnet")])
def test_state_dict_interchange_and_forward_equality(fname, ctor, ours):
    spec, a = _golden(ctor)
    mine = build_model(ours, 10)
    mine.load_state_dict(filled_state(spec), strict=True)
    mine.eval()
    with torch.no_grad():
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            b = mine(parity_input(ctor))
    assert torch.allclose(a, b, atol=2e-4, rtol=1e-4), (a - b).abs().max()


def test_transformer_matches_reference_module():
    spec, a = _golden("TransformerModel")
    mine = build_model("transformer", ntoken=1000).eval()
    mine.load_state_dict(filled_state(spec), strict=True)
    src = parity_input("TransformerModel")
    with torch.no_grad():
        b = mine(src)
    assert b.shape == (35, 3, 1000)
    assert torch.allclose(a, transformer_view(b), atol=2e-4, rtol=1e-4), (a - transformer_view(b)).abs().max()
    tgt = torch.randint(0, 1000, (35 * 3,), generator=torch.Generator().manual_seed(1))
    l1 = torch.nn.functional.nll_loss(b.view(-1, 1000), tgt)
    l2 = mine.forward_loss(src, tgt)
    assert torch.allclose(l1, l2, atol=1e-4)


def test_googlenet_fixed_order_runs_backward():
    m = build_model("googlenet", 10)
    out = m(torch.randn(2, 3, 32, 32))
    out.sum().backward()
    assert all(p.grad is not None for p in m.parameters())
