"""MNIST idx parser, DataLoader paths, CLI flag parity and an end-to-end 2-process CPU run
(ref: ddp_example.py:66-78,101-111; README.md:97-103)."""
import os
import subprocess
import sys

import pytest
import torch

import pytorch_distributed_train_b200 as pdt
from pytorch_distributed_train_b200 import cli
from pytorch_distributed_train_b200.data import (MNIST, DataLoader, DistributedSampler, SyntheticMNIST, TensorDataset,
                                                 read_idx, synthesize_mnist_files, write_idx)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_idx_roundtrip_and_mnist(tmp_path, monkeypatch):
    t = (torch.arange(2 * 28 * 28) % 251).to(torch.uint8).view(2, 28, 28)
    write_idx(str(tmp_path / "x-idx3-ubyte"), t)
    assert torch.equal(read_idx(str(tmp_path / "x-idx3-ubyte")), t)
    # an offline machine, whatever this one is: the test must never open a connection to the dataset mirrors
    monkeypatch.setattr(pdt.data.mnist, "network_reachable", lambda *a, **k: False)
    with pytest.raises(RuntimeError, match="no network is reachable"):
        MNIST(str(tmp_path / "none"), download=True)
    synthesize_mnist_files(str(tmp_path), n=300)
    ds = MNIST(str(tmp_path), train=True, download=True)
    assert len(ds) == 300
    img, y = ds[5]
    assert img.shape == (1, 28, 28) and img.dtype == torch.float32 and 0 <= img.min() and img.max() <= 1 and isinstance(y, int)
    xb, yb = ds.gather([5, 7])
    assert torch.equal(xb[0], img) and yb.dtype == torch.int64 and xb.shape == (2, 1, 28, 28)


def test_torchvision_reads_our_synthetic_files(tmp_path):
    tv = pytest.importorskip("torchvision")
    synthesize_mnist_files(str(tmp_path), n=64)
    synthesize_mnist_files(str(tmp_path), n=16, train=False)  # torchvision checks all four files
    ours = MNIST(str(tmp_path))
    theirs = tv.datasets.MNIST(str(tmp_path), train=True, transform=tv.transforms.ToTensor(), download=False)
    assert len(theirs) == 64
    a, la = ours[3]
    b, lb = theirs[3]
    assert torch.allclose(a, b) and la == lb


def test_dataloader_gather_equals_per_sample_collate():
    ds = SyntheticMNIST(250, seed=1)

    class Slow:  # same data without the batched fast path
        def __len__(self):
            return len(ds)

        def __getitem__(self, i):
            return ds[i]

    s = DistributedSampler(ds, 2, 1, shuffle=True, seed=5)
    fast = list(DataLoader(ds, batch_size=100, sampler=s))
    slow = list(DataLoader(Slow(), batch_size=100, sampler=s))
    assert len(fast) == len(slow) == 2  # 125 samples → 100 + 25
    for (xa, ya), (xb, yb) in zip(fast, slow):
        assert torch.equal(xa, xb) and torch.equal(ya, yb)
    assert fast[-1][0].shape[0] == 25
    pre = list(DataLoader(ds, batch_size=100, sampler=s, prefetch=2))
    assert all(torch.equal(a[0], b[0]) for a, b in zip(pre, fast))
    assert len(list(DataLoader(ds, batch_size=100, drop_last=True))) == 2
    td = TensorDataset(torch.arange(10.0), torch.arange(10))
    assert torch.equal(next(iter(DataLoader(td, batch_size=4)))[1], torch.arange(4))


def test_cli_flags_match_reference():
    p = cli.build_parser()
    a = p.parse_args([])
    # ref: ddp_example.py:103-106
    assert (a.gpus, a.epochs, a.backend, a.syncbn) == (1, 2, "nccl", False)
    b = p.parse_args(["-g", "4", "--epochs", "3", "--backend", "gloo", "--syncbn"])
    assert (b.gpus, b.epochs, b.backend, b.syncbn) == (4, 3, "gloo", True)
    assert a.batch_size == 100 and a.lr == 1e-4  # ref: ddp_example.py:59,62
    # the extras SURVEY §5.6 asks for, with defaults that reproduce the reference's behaviour
    assert (a.comm, a.algo, a.data, a.model, a.steps, a.graph) == ("fused", "auto", "synthetic", "convnet", 0, False)
    assert p.parse_args(["--algo", "nvls", "--comm", "nccl", "--model", "resnet18"]).algo == "nvls"


def test_train_script_two_cpu_ranks():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "train_mnist.py"), "-g", "2", "--backend", "gloo",
                          "--epochs", "1", "--steps", "20", "--samples", "4000", "--syncbn"],
                         capture_output=True, text=True, timeout=240, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    so = out.stdout
    assert "Rank id:  0" in so and "Rank id:  1" in so          # ref: ddp_example.py:49
    assert "Use SyncBN in training" in so                      # ref: ddp_example.py:56
    assert "Epoch [1/1], Step [10/20], Loss:" in so and "Epoch [1/1], Step [20/20], Loss:" in so  # ref: :94
    assert "Training complete in: " in so                      # ref: ddp_example.py:97


def test_train_script_checkpoint_and_resume(tmp_path):
    ck = str(tmp_path / "run.pt")
    base = [sys.executable, os.path.join(ROOT, "train_mnist.py"), "-g", "2", "--backend", "gloo", "--steps", "5", "--samples", "2000",
            "--log-interval", "5"]
    a = subprocess.run(base + ["--epochs", "1", "--checkpoint", ck], capture_output=True, text=True, timeout=240, cwd=ROOT)
    assert a.returncode == 0 and os.path.exists(ck), a.stderr[-2000:]
    b = subprocess.run(base + ["--epochs", "2", "--resume", ck], capture_output=True, text=True, timeout=240, cwd=ROOT)
    assert b.returncode == 0, b.stderr[-2000:]
    assert "Resumed from" in b.stdout and "Epoch [2/2], Step [5/10]" in b.stdout and "Epoch [1/2]" not in b.stdout


def test_native_batch_stager_matches_python_loader_and_never_overwrites_a_retained_batch(tmp_path):
    """_C.BatchStager (C++ worker thread + ring of staging buffers) must yield exactly what the Python loader yields,
    for the uint8 (MNIST, ToTensor's 1/255) and float32 paths, ragged last batch included — and a batch the user keeps
    (list(loader)) must never be overwritten when its ring slot comes around again (advisor finding, round 1)."""
    import pytorch_distributed_train_b200 as pdt

    pdt.data.synthesize_mnist_files(str(tmp_path), train=True, n=1030)
    m = pdt.data.MNIST(str(tmp_path), train=True)
    assert m.native_source() is not None
    for ds in (m, pdt.data.SyntheticMNIST(1030, seed=3)):
        smp = pdt.DistributedSampler(ds, num_replicas=2, rank=1, shuffle=True, seed=7)
        fast = pdt.DataLoader(ds, batch_size=100, sampler=smp)
        slow = pdt.DataLoader(ds, batch_size=100, sampler=smp, native=False)
        assert fast._native_src is not None and slow._native_src is None
        for epoch in range(2):
            smp.set_epoch(epoch)
            kept = list(fast)                      # 6 batches through an 8-slot ring, all retained
            ref = list(slow)
            assert len(kept) == len(ref) == 6 and kept[-1][0].shape[0] == 15
            for (xa, ya), (xb, yb) in zip(kept, ref):
                assert torch.allclose(xa, xb) and torch.equal(ya, yb)
    # more batches than ring slots, every one retained: earlier batches must keep their contents
    big = pdt.DataLoader(m, batch_size=10)
    kept = list(big)
    assert len(kept) == 103
    ref = list(pdt.DataLoader(m, batch_size=10, native=False))
    assert all(torch.allclose(a[0], b[0]) and torch.equal(a[1], b[1]) for a, b in zip(kept, ref))
    # a transform forces the Python path
    assert pdt.data.MNIST(str(tmp_path), train=True, transform=lambda t: t).native_source() is None


def test_native_stager_across_epochs_and_abandoned_epochs():
    """Batches are numbered across epochs inside the stager (slots waiting for CUDA events survive an epoch boundary): every epoch —
    full, shorter than the ring, or abandoned half-way — must still deliver exactly the sampler's order."""
    import torch

    from pytorch_distributed_train_b200.data import DataLoader, DistributedSampler, SyntheticMNIST

    for n, batch in ((1000, 100), (5000, 100), (730, 64)):
        ds = SyntheticMNIST(n, seed=1)
        sampler = DistributedSampler(ds, num_replicas=2, rank=1, shuffle=True, seed=5)
        loader = DataLoader(ds, batch_size=batch, sampler=sampler, prefetch=4)
        assert loader._native_src is not None
        for epoch in range(5):
            sampler.set_epoch(epoch)
            want = sampler.indices_tensor()
            got = []
            for k, (xb, yb) in enumerate(loader):
                idx = want[k * batch:(k + 1) * batch]
                assert torch.equal(xb, ds.data.index_select(0, idx)) and torch.equal(yb, ds.targets.index_select(0, idx)), (n, epoch, k)
                got.append(xb.shape[0])
                if epoch == 2 and k == 2:
                    break   # abandon this epoch: the batches staged ahead must not leak into the next one
            if epoch != 2:
                assert sum(got) == want.numel()


def test_native_stager_reports_a_worker_failure_on_the_training_thread():
    """A bad index inside the C++ gather thread must surface as an exception from next(), not abort the process."""
    import pytest
    import torch

    from pytorch_distributed_train_b200 import _C

    data = torch.zeros(10, 4, dtype=torch.uint8)
    st = _C.BatchStager(data, torch.zeros(10, dtype=torch.int64), [4], 2, False, 1.0, 4, False, -1)
    st.start(torch.tensor([0, 1, 2, 99, 4, 5], dtype=torch.int64))
    assert st.next() is not None                     # batch (0, 1) is fine
    with pytest.raises(Exception, match="out of range"):
        for _ in range(3):
            st.next()
    st.start(torch.tensor([3, 4, 5, 6], dtype=torch.int64))   # the stager is usable again after a restart
    a = st.next()
    b = st.next()
    assert a is not None and b is not None and st.next() is None
