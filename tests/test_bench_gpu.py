"""bench.py --dump-outputs on the device: the arrays written are what the op returns for the benchmark's seeded
inputs (config 1 is small enough to be written whole)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_steps_results(cuda_lib, tmp_path):
    import torch
    import surfel_scenes as S
    from diff_surfel_rasterization import GaussianRasterizationSettings, GaussianRasterizer
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "config1", "--steps", "2",
                        "--warmup", "1", "--no-cpu", "--no-e2e", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    names = ["means3D", "scales", "rotations", "opacities", "shs"]
    assert sorted(f.name for f in out.iterdir()) == sorted(
        [n + ".npy" for n in ["color", "allmap", "radii", "grad_means2D"] + [f"grad_{k}" for k in names]])

    dev = torch.device("cuda:0")
    scene, cam = S.named("config1")
    P, W, H = S.CONFIGS["config1"]
    gc, go = S.make_cotangents(W, H, S.CONFIG_SEED["config1"])
    rs = GaussianRasterizationSettings(
        image_height=H, image_width=W, tanfovx=cam["tanfovx"], tanfovy=cam["tanfovy"], bg=torch.zeros(3, device=dev),
        scale_modifier=1.0, viewmatrix=cam["viewmatrix"].to(dev), projmatrix=cam["projmatrix"].to(dev), sh_degree=3,
        campos=cam["campos"].to(dev), prefiltered=False, debug=False)
    leaf = {k: scene[k].to(dev).requires_grad_(True) for k in names}
    m2d = torch.zeros(P, 3, device=dev, requires_grad=True)
    color, radii, allmap = GaussianRasterizer(rs)(means3D=leaf["means3D"], means2D=m2d, shs=leaf["shs"],
                                                  opacities=leaf["opacities"], scales=leaf["scales"], rotations=leaf["rotations"])
    torch.autograd.backward([color, allmap], [gc.to(dev), go.to(dev)])
    load = lambda n: np.load(out / (n + ".npy"))
    for n in ("color", "allmap", "radii"):
        assert load(n).dtype == np.float32
    assert np.array_equal(load("color"), color.detach().cpu().numpy())          # the forward is bit-deterministic
    assert np.array_equal(load("allmap"), allmap.detach().cpu().numpy())
    assert np.array_equal(load("radii"), radii.cpu().numpy().astype(np.float32))
    grads = {f"grad_{k}": leaf[k].grad for k in names}
    grads["grad_means2D"] = m2d.grad
    for n, g in grads.items():                                                    # gradients: up to atomic ordering
        g = g.cpu().numpy()
        assert load(n).shape == g.shape and np.abs(load(n) - g).max() <= 1e-4 * np.abs(g).max() + 1e-30, n
