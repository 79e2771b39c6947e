"""Partitioner / corpus tests (SURVEY §4): disjoint cover, equal steps on all ranks (D8), determinism,
batchify/get_batch semantics, vocabulary size."""
import os

import numpy as np
import pytest
import torch

from dynamic_load_balance_distributeddnn_b200.data import (Corpus, DataPartitioner, batchify, get_batch,
                                                            global_permutation, load_corpus, load_image_dataset,
                                                            split_token_stream)
from dynamic_load_balance_distributeddnn_b200.data.corpus import WIKITEXT2_TOKENS, WIKITEXT2_VOCAB, SyntheticCorpus
from dynamic_load_balance_distributeddnn_b200 import ops


def test_partition_disjoint_equal_steps():
    rng = np.random.RandomState(0)
    for _ in range(50):
        n = int(rng.randint(1000, 60000))
        ws = int(rng.randint(2, 9))
        B = int(rng.choice([64, 512, 1000]))
        cuts = np.sort(rng.choice(np.arange(1, B), ws - 1, replace=False))
        lb = np.diff(np.concatenate([[0], cuts, [B]]))
        part = DataPartitioner(n, lb, seed=1234)
        allidx = np.concatenate([part.use(r).indices for r in range(ws)])
        assert len(np.unique(allidx)) == len(allidx) == part.steps * B
        assert all(part.use(r).steps == part.steps for r in range(ws))
        assert all(len(part.use(r)) == part.steps * lb[r] for r in range(ws))


def test_partition_deterministic_and_reference_permutation():
    import random
    a = DataPartitioner(5000, [40, 24], seed=1234).use(1).indices
    b = DataPartitioner(5000, [40, 24], seed=1234).use(1).indices
    assert (a == b).all()
    idx = list(range(100))
    rng = random.Random(); rng.seed(1234); rng.shuffle(idx)       # reference dataloader.py:38-40
    assert list(global_permutation(100, 1234)) == idx


def test_batchify_get_batch():
    data = torch.arange(26)
    b = batchify(data, 4)
    assert b.shape == (6, 4) and b[:, 0].tolist() == [0, 1, 2, 3, 4, 5] and b[0].tolist() == [0, 6, 12, 18]
    x, y = get_batch(b, 0, 3)
    assert x.shape == (3, 4) and y.tolist() == b[1:4].reshape(-1).tolist()
    x, y = get_batch(b, 3, 35)
    assert x.shape == (2, 4)                                          # clipped at the end


def test_token_stream_split_equal_rows():
    pieces = split_token_stream(2088628, [22, 21, 21])
    rows = [(p.stop - p.start) // b for p, b in zip(pieces, [22, 21, 21])]
    assert len(set(rows)) == 1 and pieces[0].start == 0 and pieces[1].start == pieces[0].stop


def test_corpus_tokenize(tmp_path):
    for name, txt in (("train", "a b c\nb c d\n"), ("valid", "a e\n"), ("test", "f\n")):
        (tmp_path / f"{name}.txt").write_text(txt)
    c = Corpus(str(tmp_path))
    assert c.ntokens == 7                                             # a b c <eos> d e f
    assert c.train.tolist() == [0, 1, 2, 3, 1, 2, 4, 3]
    s = SyntheticCorpus(vocab=100, sizes={"train": 1000, "valid": 100, "test": 100})
    assert s.ntokens == 100 and int(s.train.max()) == 99


def test_wikitext2_vocab(monkeypatch, tmp_path):
    """tests/golden/wikitext2_sample holds the first lines of each wikitext-2 split; wikitext2_sample.npz the token ids and
    vocabulary size the reference's Corpus produced for them, and its vocabulary size and split lengths on the full corpus
    (the shape the synthetic stand-in copies)."""
    golden = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    ref = np.load(os.path.join(golden, "wikitext2_sample.npz"))
    monkeypatch.setenv("DLB_CACHE_DIR", str(tmp_path))
    c = load_corpus(os.path.join(golden, "wikitext2_sample"))
    assert c.ntokens == int(ref["ntokens"])
    for split in ("train", "valid", "test"):
        assert getattr(c, split).tolist() == ref[split].tolist(), split
    full = ref["full"].tolist()
    assert full == [WIKITEXT2_VOCAB, WIKITEXT2_TOKENS["train"], WIKITEXT2_TOKENS["valid"], WIKITEXT2_TOKENS["test"]]


def test_synthetic_images_and_augment():
    ds = load_image_dataset("cifar10", True, synthetic=True, n_override=256)
    assert ds.images.shape == (256, 32, 32, 3) and ds.images.dtype == torch.uint8 and ds.labels.max() < 10
    x = ops.augment(ds.images[:8], ds.mean, ds.std, ds.pad, ds.flip, seed=3, step=5, dtype=torch.float32)
    assert x.shape == (8, 3, 32, 32) and x.stride(1) == 1            # channels-last memory
    x0 = ops.augment(ds.images[:8], ds.mean, ds.std, 0, False, dtype=torch.float32)
    ref = (ds.images[:8].float() / 255 - torch.tensor(ds.mean)) / torch.tensor(ds.std)
    assert torch.allclose(x0.permute(0, 2, 3, 1), ref, atol=1e-6)
    t = load_image_dataset("mnist", False, synthetic=True, n_override=64)
    assert t.images.shape == (64, 28, 28, 1) and t.pad == 0


def test_partitioner_segments_cover_one_permutation():
    """--rebalance_every: segments with different splits still form a disjoint cover of the epoch's permutation."""
    from dynamic_load_balance_distributeddnn_b200.data import DataPartitioner
    n, seen, used = 1000, [], 0
    for lbs in ([16, 16], [20, 12], [25, 7]):
        p = DataPartitioner(n, lbs, 1234, True, 5, start=used)
        assert p.steps == 5
        for r in range(2):
            seen += list(p.use(r).indices)
        used += p.steps * 32
    assert len(seen) == len(set(seen)) == 3 * 5 * 32


def test_real_dataset_files_are_used_when_present(tmp_path):
    """A pre-populated torchvision layout (here: FashionMNIST raw idx files, which the reference's `-ds mnist` reads) is
    loaded instead of the synthetic stand-in; `--synthetic false` without files fails loudly."""
    import struct
    pytest.importorskip("torchvision")
    from dynamic_load_balance_distributeddnn_b200.data import vision
    raw = tmp_path / "FashionMNIST" / "raw"
    raw.mkdir(parents=True)
    rng = np.random.RandomState(0)

    def write(prefix, n):
        img = rng.randint(0, 256, size=(n, 28, 28), dtype=np.uint8)
        lab = rng.randint(0, 10, size=(n,), dtype=np.uint8)
        (raw / f"{prefix}-images-idx3-ubyte").write_bytes(struct.pack(">IIII", 0x00000803, n, 28, 28) + img.tobytes())
        (raw / f"{prefix}-labels-idx1-ubyte").write_bytes(struct.pack(">II", 0x00000801, n) + lab.tobytes())
        return img, lab
    img, lab = write("train", 48)
    write("t10k", 16)
    ds = vision.load_image_dataset("mnist", True, root=str(tmp_path), synthetic=False)
    assert not ds.synthetic and tuple(ds.images.shape) == (48, 28, 28, 1) and ds.images.dtype == torch.uint8
    assert np.array_equal(ds.images[..., 0].numpy(), img) and np.array_equal(ds.labels.numpy(), lab.astype(np.int64))
    assert len(vision.load_image_dataset("mnist", False, root=str(tmp_path), synthetic=None).labels) == 16
    with pytest.raises(FileNotFoundError):
        vision.load_image_dataset("cifar10", True, root=str(tmp_path / "nothing"), synthetic=False)
