"""Drop-in evidence against the reference's own Python, through data it produced (tests/golden/ref_interop.npz,
written by tests/golden/make_golden_interop.py from a checkout of the reference).

  * The reference's densification code (training_setup, update_learning_rate, prune_points, densification_postfix,
    reset_opacity, capture) manipulates its optimizer only through the torch.optim.Adam surface: it selects rows of
    a group's parameter and of its Adam moments, appends rows with zero moments, and replaces a parameter with its
    moments zeroed, each time re-keying optimizer.state to the new nn.Parameter.  The golden holds the optimizer as
    that code left a torch.optim.Adam; the same operations applied to `diff_surfel_rasterization.optim.FusedAdam`
    must leave it in exactly that state.  (FusedAdam.step itself needs a GPU and is covered by
    tests/test_optim_gpu.py; here the per-parameter state is planted by hand, as Adam would create it.)
  * The reference's unmodified gaussian_renderer.render() passes fixed keyword patterns to
    GaussianRasterizationSettings(...) and GaussianRasterizer(...)(...) (compute_cov3D_python on/off x SH /
    override_color inputs); the golden holds them verbatim and they must drive OUR Python surface down to the
    native call, which is replaced here (no GPU)."""
import json
import os

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "ref_interop.npz")


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


def _optimizer_as_the_reference_leaves_it(adam_cls, gold):
    names = [str(n) for n in gold["opt_names"]]
    lr0, eps = (float(x) for x in gold["opt_defaults"])
    params = [torch.nn.Parameter(torch.from_numpy(gold[f"opt_init_{n}_param"].copy())) for n in names]
    opt = adam_cls([{"params": [p], "lr": float(lr), "name": n} for p, lr, n in zip(params, gold["opt_init_lr"], names)],
                   lr=lr0, eps=eps)
    for grp in opt.param_groups:                                       # state as Adam creates it on the first step
        n = grp["name"]
        opt.state[grp["params"][0]] = {"step": torch.tensor(3.0),
                                       "exp_avg": torch.from_numpy(gold[f"opt_init_{n}_exp_avg"].copy()),
                                       "exp_avg_sq": torch.from_numpy(gold[f"opt_init_{n}_exp_avg_sq"].copy())}

    def swap(grp, param_fn, moment_fn):
        old = grp["params"][0]
        st = opt.state.pop(old)
        for k in ("exp_avg", "exp_avg_sq"):
            st[k] = moment_fn(st[k])
        grp["params"][0] = torch.nn.Parameter(param_fn(old.detach()).requires_grad_(True))
        opt.state[grp["params"][0]] = st

    for grp in opt.param_groups:                                       # update_learning_rate: the xyz group only
        if grp["name"] == "xyz":
            grp["lr"] = float(gold["opt_xyz_lr"])
    keep = torch.from_numpy(~gold["opt_prune_mask"])
    for grp in opt.param_groups:                                       # prune_points
        swap(grp, lambda t: t[keep], lambda m: m[keep])
    for grp in opt.param_groups:                                       # densification_postfix
        ext = torch.from_numpy(gold[f"opt_append_{grp['name']}"].copy())
        swap(grp, lambda t: torch.cat((t, ext)), lambda m: torch.cat((m, torch.zeros_like(ext))))
    for grp in opt.param_groups:                                       # reset_opacity
        if grp["name"] == "opacity":
            new = torch.from_numpy(gold["opt_final_opacity_param"].copy())
            swap(grp, lambda t: new, torch.zeros_like)
    return opt


def test_reference_densification_code_runs_unchanged_on_fused_adam(gold):
    from diff_surfel_rasterization.optim import FusedAdam
    arms = {cls.__name__: _optimizer_as_the_reference_leaves_it(cls, gold) for cls in (torch.optim.Adam, FusedAdam)}
    assert isinstance(arms["FusedAdam"], torch.optim.Adam)
    for arm, opt in arms.items():            # torch's own Adam as well: the replay itself must reproduce the reference
        assert [g["name"] for g in opt.param_groups] == [str(n) for n in gold["opt_names"]], arm
        for grp in opt.param_groups:
            n, p = grp["name"], grp["params"][0]
            assert grp["lr"] == float(gold[f"opt_final_{n}_lr"]) and grp["eps"] == float(gold[f"opt_final_{n}_eps"]) == 1e-15
            assert tuple(grp["betas"]) == tuple(gold[f"opt_final_{n}_betas"]), (arm, n)
            assert p.shape[0] == 12 - 3 + 4 and torch.equal(p.detach(), torch.from_numpy(gold[f"opt_final_{n}_param"])), (arm, n)
            st = opt.state[p]
            assert set(st) == {"step", "exp_avg", "exp_avg_sq"}, (arm, n)
            for k in st:
                assert torch.equal(st[k], torch.from_numpy(np.asarray(gold[f"opt_final_{n}_{k}"]))), (arm, n, k)
    sd_ref = arms["Adam"].state_dict()
    sd_fused = arms["FusedAdam"].state_dict()                          # capture(): optimizer.state_dict()
    assert {str(k) for k in gold["opt_state_dict_group_keys"]} <= set(sd_fused["param_groups"][0])
    assert set(sd_ref["param_groups"][0]) <= set(sd_fused["param_groups"][0])
    arms["FusedAdam"].load_state_dict(sd_ref)                          # a checkpoint written with torch's Adam loads


def _replayed(gold, i, part, meta):
    kw = {}
    for k, m in meta.items():
        if m["kind"] == "tensor":
            t = torch.from_numpy(np.asarray(gold[f"render{i}_{part}_{k}"]).copy())
            assert str(t.dtype).replace("torch.", "") == m["dtype"], k
            kw[k] = t.requires_grad_(m["requires_grad"])
        else:
            kw[k] = m["value"]
    return kw


def test_reference_render_drives_our_python_surface(gold, monkeypatch):
    """Our GaussianRasterizationSettings and GaussianRasterizer accept the reference render()'s own keywords and
    argument patterns; only the native call below the Python surface is replaced."""
    import diff_surfel_rasterization as real
    calls = []

    def fake_native(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, rs):
        calls.append(dict(means3D=means3D, means2D=means2D, sh=sh, colors_precomp=colors_precomp, opacities=opacities,
                          scales=scales, rotations=rotations, cov3Ds_precomp=cov3Ds_precomp, rs=rs))
        H, W = rs.image_height, rs.image_width
        return torch.zeros(3, H, W), torch.ones(means3D.shape[0], dtype=torch.int32), torch.ones(7, H, W)
    monkeypatch.setattr(real, "rasterize_gaussians", fake_native)
    meta = json.loads(str(gold["render_meta"]))
    assert [(m["cov3D_python"], m["override_color"]) for m in meta] == [(False, False), (False, True), (True, False), (True, True)]
    for i, m in enumerate(meta):
        cov_py, sh_py = m["cov3D_python"], m["override_color"]
        rs_in = real.GaussianRasterizationSettings(**_replayed(gold, i, "settings", m["settings"]))
        color, radii, allmap = real.GaussianRasterizer(raster_settings=rs_in)(**_replayed(gold, i, "call", m["call"]))
        c = calls[-1]
        rs = c["rs"]
        P = c["means3D"].shape[0]
        H, W = rs.image_height, rs.image_width
        assert isinstance(rs, real.GaussianRasterizationSettings)
        assert (H, W, rs.sh_degree, rs.prefiltered, rs.scale_modifier) == (48, 64, 3, False, 1.0)
        assert isinstance(rs.tanfovx, float) and rs.viewmatrix.shape == (4, 4) and rs.projmatrix.shape == (4, 4) and rs.campos.shape == (3,)
        assert P == 10 and c["means2D"].shape == (P, 3) and c["opacities"].shape == (P, 1)
        assert (c["cov3Ds_precomp"].numel() > 0) == cov_py and (c["scales"].numel() > 0) == (not cov_py) and (c["rotations"].numel() > 0) == (not cov_py)
        assert (c["colors_precomp"].numel() > 0) == sh_py and (c["sh"].numel() > 0) == (not sh_py)
        if cov_py:
            assert c["cov3Ds_precomp"].shape == (P, 9)
        if not sh_py:
            assert c["sh"].shape == (P, 16, 3)
        assert color.shape == (3, H, W) and allmap.shape == (7, H, W) and radii.shape == (P,) and radii.dtype == torch.int32
    assert len(calls) == 4
