"""bench.py --dump-outputs: one float32 file per output and per parameter gradient; an array above
its size cap becomes the same seeded sample in every run, so two builds compare file for file."""
import numpy as np
import torch

import bench


def test_dump_outputs_writes_float32_files_and_a_fixed_sample(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_GRAD_ELEMS", 64)
    model = torch.nn.Linear(16, 8)
    for p in model.parameters():
        p.grad = torch.randn_like(p)
    clip = torch.randn(2, 5, 8).bfloat16()
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"clip": clip}, model)
    names = sorted(f.name for f in (tmp_path / "a").iterdir())
    assert names == ["clip.npy", "grad.bias.npy", "grad.weight.npy"]
    a = {n: np.load(tmp_path / "a" / n) for n in names}
    assert all(x.dtype == np.float32 for x in a.values())
    assert np.array_equal(a["clip.npy"], clip.float().numpy())
    assert np.array_equal(a["grad.bias.npy"], model.bias.grad.numpy())
    w = a["grad.weight.npy"]                      # 128 elements > cap: a sample of 64 of them
    assert w.shape == (64,) and np.isin(w, model.weight.grad.numpy()).all()
    assert np.array_equal(w, np.load(tmp_path / "b" / "grad.weight.npy"))
