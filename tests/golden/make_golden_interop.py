"""Generates tests/golden/ref_interop.npz by running the reference's own Python on the CPU (needs a checkout of
the reference; its path is the first argument).  tests/test_reference_interop_cpu.py compares against it.

  optimizer: the reference's GaussianModel.training_setup builds its optimizer with torch.optim.Adam; with the
    per-parameter state planted as Adam creates it on its first step, update_learning_rate(1000), prune_points,
    densification_postfix and reset_opacity run unchanged.  Stored: the groups and state after training_setup
    (opt_init_*), the prune mask, the appended rows, the xyz learning rate, and every group's parameter and
    state at the end (opt_final_*).
  render: the reference's unmodified gaussian_renderer.render() is run against a capturing stand-in of
    diff_surfel_rasterization for compute_cov3D_python in {False, True} x {SH, override_color}.  Stored: the
    keyword arguments it passes to GaussianRasterizationSettings(...) and to GaussianRasterizer(...)(...).

Usage:  python tests/golden/make_golden_interop.py <path of the reference checkout>
"""
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "2d-gaussian-splatting_b200"))


def optimizer_fixture(GM, out):
    g = torch.Generator("cpu").manual_seed(5)
    P = 12
    pc = GM.GaussianModel(3)
    pc._xyz = torch.nn.Parameter(torch.randn(P, 3, generator=g))
    pc._features_dc = torch.nn.Parameter(torch.randn(P, 1, 3, generator=g))
    pc._features_rest = torch.nn.Parameter(torch.randn(P, 15, 3, generator=g))
    pc._opacity = torch.nn.Parameter(torch.randn(P, 1, generator=g))
    pc._scaling = torch.nn.Parameter(torch.randn(P, 2, generator=g))
    pc._rotation = torch.nn.Parameter(torch.randn(P, 4, generator=g))
    pc.max_radii2D = torch.zeros(P)
    pc.spatial_lr_scale = 5.0
    args = types.SimpleNamespace(percent_dense=0.01, position_lr_init=0.00016, position_lr_final=0.0000016,
                                 position_lr_delay_mult=0.01, position_lr_max_steps=30000, feature_lr=0.0025,
                                 opacity_lr=0.05, scaling_lr=0.005, rotation_lr=0.001)
    pc.training_setup(args)
    opt = pc.optimizer
    assert type(opt) is torch.optim.Adam
    names = [grp["name"] for grp in opt.param_groups]
    out["opt_names"] = np.array(names)
    out["opt_init_lr"] = np.array([grp["lr"] for grp in opt.param_groups], np.float64)
    out["opt_defaults"] = np.array([opt.defaults["lr"], opt.defaults["eps"]], np.float64)
    for grp in opt.param_groups:
        p = grp["params"][0]
        opt.state[p] = {"step": torch.tensor(3.0), "exp_avg": torch.randn(p.shape, generator=g),
                        "exp_avg_sq": torch.rand(p.shape, generator=g)}
        n = grp["name"]
        out[f"opt_init_{n}_param"] = p.detach().numpy().copy()
        out[f"opt_init_{n}_exp_avg"] = opt.state[p]["exp_avg"].numpy().copy()
        out[f"opt_init_{n}_exp_avg_sq"] = opt.state[p]["exp_avg_sq"].numpy().copy()
    out["opt_xyz_lr"] = np.float64(pc.update_learning_rate(1000))
    mask = torch.zeros(P, dtype=torch.bool)
    mask[[1, 4, 9]] = True
    out["opt_prune_mask"] = mask.numpy()
    pc.prune_points(mask)
    n = 4
    new = {"xyz": torch.ones(n, 3), "f_dc": torch.ones(n, 1, 3), "f_rest": torch.ones(n, 15, 3),
           "opacity": torch.ones(n, 1), "scaling": torch.ones(n, 2), "rotation": torch.ones(n, 4)}
    pc.densification_postfix(*(new[k] for k in ("xyz", "f_dc", "f_rest", "opacity", "scaling", "rotation")))
    for k, v in new.items():
        out[f"opt_append_{k}"] = v.numpy()
    pc.reset_opacity()
    sd = pc.capture()[-2]                                              # optimizer.state_dict() inside capture()
    out["opt_state_dict_group_keys"] = np.array(sorted(sd["param_groups"][0]))
    for grp in opt.param_groups:
        p, st, n = grp["params"][0], opt.state[grp["params"][0]], grp["name"]
        assert set(st) == {"step", "exp_avg", "exp_avg_sq"}
        out[f"opt_final_{n}_lr"] = np.float64(grp["lr"])
        out[f"opt_final_{n}_betas"] = np.array(grp["betas"], np.float64)
        out[f"opt_final_{n}_eps"] = np.float64(grp["eps"])
        out[f"opt_final_{n}_param"] = p.detach().numpy().copy()
        for k in ("step", "exp_avg", "exp_avg_sq"):
            out[f"opt_final_{n}_{k}"] = st[k].numpy().copy()


def render_fixture(ref, out):
    import surfel_scenes as S
    calls = []

    class Settings:
        def __init__(self, **kw):
            self.kw = kw

    class Rasterizer:
        def __init__(self, raster_settings):
            self.rs = raster_settings

        def __call__(self, **kw):
            calls.append((self.rs.kw, kw))
            H, W = self.rs.kw["image_height"], self.rs.kw["image_width"]
            return torch.zeros(3, H, W), torch.ones(kw["means3D"].shape[0], dtype=torch.int32), torch.ones(7, H, W)
    dsr = sys.modules["diff_surfel_rasterization"]
    dsr.GaussianRasterizationSettings, dsr.GaussianRasterizer = Settings, Rasterizer
    sys.path.insert(0, ref)
    from gaussian_renderer import render
    from scene.cameras import Camera
    from scene.gaussian_model import GaussianModel

    W, H, P = 64, 48, 10
    Rm, tv = S.look_at_rotation(10, 5), np.array([0.1, 0.0, 0.3])
    mycam = S.make_camera(W, H, R=Rm, t=tv)
    cam = Camera(colmap_id=0, R=Rm, T=tv, FoVx=mycam["FoVx"], FoVy=mycam["FoVy"], image=torch.zeros(3, H, W),
                 gt_alpha_mask=None, image_name="g", uid=0, data_device="cpu")
    scene = S.make_scene(P, W, H, 4, depth_complexity=2)
    pc = GaussianModel(3)
    pc.active_sh_degree = 3
    pc._xyz, pc._scaling, pc._rotation = scene["means3D"], torch.log(scene["scales"]), scene["rotations"]
    pc._opacity = torch.log(scene["opacities"] / (1 - scene["opacities"]))
    pc._features_dc, pc._features_rest = scene["shs"][:, :1].contiguous(), scene["shs"][:, 1:].contiguous()
    g = torch.Generator("cpu").manual_seed(7)
    meta = []
    for cov_py in (False, True):
        for sh_py in (False, True):
            pipe = types.SimpleNamespace(compute_cov3D_python=cov_py, convert_SHs_python=False, depth_ratio=0.0, debug=False)
            render(cam, pc, pipe, torch.zeros(3), override_color=torch.rand(P, 3, generator=g) if sh_py else None)
            i = len(meta)
            entry = {"cov3D_python": cov_py, "override_color": sh_py, "settings": {}, "call": {}}
            for part, kw in zip(("settings", "call"), calls[-1]):
                for k, v in kw.items():
                    if isinstance(v, torch.Tensor):
                        out[f"render{i}_{part}_{k}"] = v.detach().numpy().copy()
                        entry[part][k] = {"kind": "tensor", "dtype": str(v.dtype).replace("torch.", ""),
                                          "requires_grad": v.requires_grad}
                    else:
                        entry[part][k] = {"kind": type(v).__name__, "value": v}
            meta.append(entry)
    assert len(calls) == 4
    out["render_meta"] = np.array(json.dumps(meta))


def main():
    ref = os.path.abspath(sys.argv[1])
    import make_golden as MG
    MG.cpu_patches()
    MG.stub_modules({})
    sys.path.insert(0, ref)
    import scene.gaussian_model as GM
    out = {}
    optimizer_fixture(GM, out)
    render_fixture(ref, out)
    np.savez_compressed(os.path.join(HERE, "ref_interop.npz"), **out)
    print("wrote ref_interop.npz:", len(out), "arrays")


if __name__ == "__main__":
    main()
