#!/usr/bin/env python
"""Record what the reference-parity tests compare against, from a checkout of the reference project, into tests/golden/:

    python tools/make_golden.py /path/to/reference

* model_parity.json / .npz  -- state_dict layout of the reference's Net/* classes and their outputs on a seeded input in a
                               state that depends only on that layout (tests/test_models.py);
* gradpath.npz              -- loss and a stratified gradient sample of one fp32 step of the reference's models on the
                               weights and images our trainer starts from (tests/test_gpu_gradpath.py);
* wikitext2_sample/ + .npz  -- the first lines of each wikitext-2 split and the reference Corpus' token ids for them, plus its
                               vocabulary size and split lengths on the full corpus (tests/test_data.py).

Runs on the CPU; the reference is imported from its own directory and nothing of it is copied except corpus lines.
"""
import importlib.util
import json
import os
import sys
import tempfile

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from test_gpu_gradpath import gradient_sample                             # noqa: E402
from test_models import filled_state, parity_input, transformer_view      # noqa: E402

CORPUS_LINES = 60


def ref_module(ref, rel):
    spec = importlib.util.spec_from_file_location("ref_" + rel.replace("/", "_")[:-3], os.path.join(ref, rel))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def model_parity(ref):
    layouts, outs = {}, {}
    for fname, ctor in (("Densenet.py", "DenseNet121"), ("Resnet.py", "ResNet50"), ("Resnet.py", "ResNet18"),
                        ("RegNet.py", "RegNetY_400MF"), ("MnistNet.py", "MnistNet"), ("Transformer.py", "TransformerModel")):
        mod = ref_module(ref, "Net/" + fname)
        if ctor == "MnistNet":
            m = mod.MnistNet()
        elif ctor == "TransformerModel":
            m = mod.TransformerModel(1000, 200, 2, 200, 2, 0.2)
        else:
            m = getattr(mod, ctor)(10)
        spec = [(k, list(v.shape), str(v.dtype).replace("torch.", "")) for k, v in m.state_dict().items()]
        m.load_state_dict(filled_state([(k, tuple(s), d) for k, s, d in spec]), strict=True)
        m.eval()
        with torch.no_grad():
            out = m(parity_input(ctor))
        layouts[ctor] = spec
        outs[ctor] = (transformer_view(out) if ctor == "TransformerModel" else out).numpy().astype(np.float32)
    with open(os.path.join(GOLDEN, "model_parity.json"), "w") as f:
        f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(v, separators=(',', ':'))}" for k, v in layouts.items()) + "\n}\n")
    np.savez_compressed(os.path.join(GOLDEN, "model_parity.npz"), **outs)


def gradpath(ref):
    from dynamic_load_balance_distributeddnn_b200.config import DBSConfig
    from dynamic_load_balance_distributeddnn_b200.engine import Trainer
    from dynamic_load_balance_distributeddnn_b200.utils import init_logger
    out = {}
    cases = [("densenet", "Densenet", "DenseNet121", "tf32"), ("densenet", "Densenet", "DenseNet121", "bf16"),
             ("resnet18", "Resnet", "ResNet18", "bf16"), ("resnet50", "Resnet", "ResNet50", "bf16"),
             ("regnet", "RegNet", "RegNetY_400MF", "bf16"), ("resnet18", "Resnet", "ResNet18", "tf32"),
             ("regnet", "RegNet", "RegNetY_400MF", "tf32")]
    with tempfile.TemporaryDirectory() as tmp:
        for model, ref_mod, ref_cls, dtype in cases:
            # the trainer of tests/test_gpu_gradpath.py::_trainer, built on the CPU: same initial weights and images
            cfg = DBSConfig(debug=False, world_size=1, batch_size=16, model=model, dataset="cifar10", synthetic=True,
                            train_samples=16 * 8, test_samples=64, epoch_size=1, validate=False, cuda_graphs=False, dtype=dtype,
                            learning_rate=0.05, log_dir=os.path.join(tmp, "l"), stats_dir=os.path.join(tmp, "s"))
            t = Trainer(cfg, 0, 1, "cpu", init_logger(cfg, 0, stream=False))
            t.train_set.pad, t.train_set.flip = 0, False
            xb, yb = t.stager.stage(list(range(16)))
            x = t._prepare_images(xb).float()
            m = getattr(ref_module(ref, f"Net/{ref_mod}.py"), ref_cls)(10).float()
            m.load_state_dict({k: v.detach().float().clone() for k, v in t.model.state_dict().items()})
            loss = F.cross_entropy(m(x.contiguous()), yb)
            loss.backward()
            params = [p for _, p in t.model.named_parameters()]
            grads = [p.grad for _, p in m.named_parameters()]
            ti, ei = gradient_sample([p.numel() for p in params])
            pick = lambda ts: np.concatenate([ts[i].detach().float().reshape(-1)[torch.as_tensor(ei[ti == i])].numpy()  # noqa: E731
                                              for i in range(len(ts))])
            pre = f"{model}-{dtype}/"
            out.update({pre + "numel": np.array([p.numel() for p in params]), pre + "w0": pick(params), pre + "grad": pick(grads),
                        pre + "loss": np.float64(loss.item()), pre + "labels": yb.numpy().astype(np.int8),
                        pre + "x_sum": np.float64(x.double().sum().item())})
            print(pre, "loss", loss.item(), flush=True)
    np.savez_compressed(os.path.join(GOLDEN, "gradpath.npz"), **out)


def corpus(ref):
    mod = ref_module(ref, "dataloader.py")
    src = os.path.join(ref, "rnn_data", "wikitext-2")
    full = mod.Corpus(src)
    dst = os.path.join(GOLDEN, "wikitext2_sample")
    os.makedirs(dst, exist_ok=True)
    for split in ("train", "valid", "test"):
        with open(os.path.join(src, split + ".txt"), encoding="utf8") as f:
            lines = [next(f) for _ in range(CORPUS_LINES)]
        with open(os.path.join(dst, split + ".txt"), "w", encoding="utf8") as f:
            f.writelines(lines)
    sample = mod.Corpus(dst)
    np.savez_compressed(os.path.join(GOLDEN, "wikitext2_sample.npz"), ntokens=len(sample.dictionary),
                        train=sample.train.numpy().astype(np.int32), valid=sample.valid.numpy().astype(np.int32),
                        test=sample.test.numpy().astype(np.int32),
                        full=np.array([len(full.dictionary), full.train.numel(), full.valid.numel(), full.test.numel()]))


if __name__ == "__main__":
    ref = os.path.realpath(sys.argv[1])
    os.makedirs(GOLDEN, exist_ok=True)
    torch.manual_seed(0)
    model_parity(ref)
    corpus(ref)
    gradpath(ref)
