"""The torch-op comparator that bench.py times beside the CUDA path (baseline/torch_reference_path.py) must BE the
reference's formulation: on the same skeleton with the same random draws it reproduces, bit for bit, the output of the
reference's own patched UNet, stored in tests/golden/restatement_tiny_f*.npz by `tests/make_golden_r02.py --restatement`."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("frames", [4, 8])
def test_restatement_equals_reference_on_cpu(frames, monkeypatch):
    sys.path.insert(0, ROOT)
    from baseline import torch_reference_path as R
    from vidtome_b200.skeleton import make_skeleton
    g = np.load(os.path.join(ROOT, "tests", "golden", f"restatement_tiny_f{frames}.npz"))
    draws = iter(g["draws"].tolist())

    def fixed(lo, hi, size, **kw):
        v = next(draws) % hi
        return torch.full(tuple(size), v, dtype=torch.int64)
    x = torch.from_numpy(g["x"])
    net = make_skeleton("tiny", device="cpu", dtype=torch.float32, hot_path_only=False, seed=5)
    monkeypatch.setattr(torch, "randint", fixed)
    # the reference's CPU argsort is not stable; the fixture was made with the (CUDA-like) stable order
    real_argsort = torch.Tensor.argsort
    monkeypatch.setattr(torch.Tensor, "argsort", lambda t, *a, **k: real_argsort(t, *a, **{**k, "stable": True}))
    R.apply_reference_path(net, 0.9, 2)
    with torch.no_grad():
        out = net(x, 0, encoder_hidden_states=torch.zeros(2 * frames, 7, 768)).sample
    assert torch.equal(out, torch.from_numpy(g["out"]))


def test_config1_plumbing_on_cpu():
    """BASELINE config 1 as the reference defines it (device=cpu, 4 frames, 10 DDIM steps, local merge only: plumbing,
    no GPU): the reference formulation (baseline/torch_reference_path.py, the CPU arm of bench.py) through the chunked
    DDIM driver on the CPU in fp32.  The CUDA package itself has no CPU path by design."""
    sys.path.insert(0, ROOT)
    from baseline import torch_reference_path as R
    from vidtome_b200.driver import ChunkedDenoiser
    from vidtome_b200.skeleton import make_skeleton
    net = make_skeleton("tiny", device="cpu", dtype=torch.float32, hot_path_only=False, seed=4)
    R.apply_reference_path(net, 0.95, 2)
    den = ChunkedDenoiser(net, n_timesteps=10, chunk_size=4, cond=torch.randn(2, 7, 768))
    torch.manual_seed(0)
    x = den.sample(torch.randn(4, 4, 16, 16))
    assert x.shape == (4, 4, 16, 16) and torch.isfinite(x).all()
    R.remove_reference_path(net)
