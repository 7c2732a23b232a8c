"""bench.py's ``--dump-outputs``: the arrays it writes are the last timed step's energy and forces, within the size limit."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_caps_forces_at_a_fixed_sample_of_rows(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4096 + 4 + 12 * 100)
    grad = torch.arange(3000, dtype=torch.float32).reshape(1000, 3)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), torch.tensor([1.5]), grad)
    fa, fb = np.load(tmp_path / "a" / "forces.npy"), np.load(tmp_path / "b" / "forces.npy")
    assert fa.shape == (100, 3) and fa.dtype == np.float32
    assert np.array_equal(fa, fb)
    rows = -fa[:, 0] / 3
    assert np.array_equal(rows, np.unique(rows)) and np.array_equal(fa, -grad.numpy()[rows.astype(np.int64)])
    assert np.load(tmp_path / "a" / "energy.npy").tolist() == [1.5]
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in ("energy.npy", "forces.npy")) <= bench.DUMP_LIMIT_BYTES


@pytest.mark.gpu
def test_dump_outputs_are_the_energy_and_forces_of_the_timed_step(tmp_path):
    import hermnet_b200 as H
    from hermnet_b200 import synthetic
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1", "--scale", "0.1",
           "--e2e-steps", "0", "--no-cpu-baseline", "--no-parity", "--dump-outputs", str(tmp_path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2
    e, f = np.load(tmp_path / "energy.npy"), np.load(tmp_path / "forces.npy")

    (pos, Z, cell), cfg = synthetic.config("C4", 0.1)
    kind = cfg.pop("kind")
    torch.manual_seed(1234)
    model = getattr(H, kind)(**cfg).cuda().eval()
    for p in model.parameters():
        p.requires_grad_(False)
    d = H.Data(pos=torch.from_numpy(pos).cuda().requires_grad_(True), atomic_number=torch.from_numpy(Z).cuda(),
               cell=torch.from_numpy(cell)[None].cuda())
    e_ref = model(d)
    (g,) = torch.autograd.grad(e_ref.sum(), d.pos)
    e_ref, f_ref = e_ref.detach().cpu().numpy(), -g.cpu().numpy()
    assert e.dtype == np.float32 and e.shape == e_ref.shape and f.dtype == np.float32 and f.shape == (len(Z), 3)
    assert np.abs(e - e_ref).max() <= 1e-5 * np.abs(e_ref).max()
    assert np.abs(f - f_ref).max() <= 1e-4 * max(1.0, np.abs(f_ref).max())
