"""End-to-end: ngp_pl_b200's render()/NGP against the UNMODIFIED reference render()/NGP (driven by the reference's
compiled vren + the tinycudann stand-in) on identical rays, identical weights, identical start jitter (same torch seed
-> same torch.rand_like draw). The reference's results are stored in tests/golden/parity_render.npz
(tests/golden/make_golden_parity.py).

  marcher        : rm_samples and per-ray sample counts identical
  rgb/depth/opac : the network part is only pinned to fp16 level (tinycudann is absent), so the
                   rendered values agree to ~1e-3 absolute; given IDENTICAL sigmas/rgbs the compositor
                   agrees to 1e-4 relative (tests/test_vren_gpu.py).
"""
import numpy as np
import pytest
import torch

import cases

pytestmark = pytest.mark.gpu


def _rays(scene, n, seed):
    o, d = cases.rays_from_scene(scene, n, seed, extra_edge_cases=False)
    return torch.as_tensor(o).cuda(), torch.as_tensor(d).cuda()


@pytest.mark.parametrize("which", ["lego", "mip360"])
def test_train_render_matches_reference(which):
    from ngp_pl_b200.losses import NeRFLoss
    from ngp_pl_b200.models.rendering import render
    g = cases.golden("parity_render.npz")
    pre = "render_%s_" % which
    scene = cases.scene_by_name(which)
    mine = cases.seeded_ngp(scene)
    o, d = _rays(scene, 2048, 31)
    kw = {} if scene.exp_step_factor == 0 else {"exp_step_factor": scene.exp_step_factor}
    torch.manual_seed(123)
    r_my = render(mine, o, d, **kw)
    assert int(g[pre + "rm_samples"]) == int(r_my["rm_samples"]) > 0
    assert (g[pre + "counts"] == r_my["rays_a"][:, 2].cpu().numpy()).all()
    for k in ("rgb", "opacity", "depth"):
        ref_k = g[pre + k]
        err = np.abs(ref_k - r_my[k].detach().float().cpu().numpy()).max()
        assert err < 5e-3 * max(1.0, np.abs(ref_k).max()), "%s differs by %g" % (k, err)
    for k in g[pre + "keys"]:
        assert k in r_my, "missing result key " + k

    # gradients of the reference's loss (NeRFLoss, no distortion term) through both pipelines
    mine.zero_grad()
    l = NeRFLoss(lambda_distortion=0)(r_my, {"rgb": cases.render_target(o.shape[0])})
    sum(v.mean() for v in l.values()).backward()
    cases.check_grads_vs_golden(mine, g, pre, 0.06)


def test_test_render_matches_reference():
    from ngp_pl_b200 import synth
    from ngp_pl_b200.models.rendering import render
    g = cases.golden("parity_render.npz")
    scene = synth.lego_scene(0)
    mine = cases.seeded_ngp(scene)
    K = synth.intrinsics(W=100, H=100, fx=1111.11 / 8)
    dirs = synth.ray_directions(K, "cuda")
    pose = torch.as_tensor(synth.camera_poses(3)[2]).cuda()
    o, d = synth.get_rays(dirs, pose)
    r_my = render(mine, o, d, test_time=True)
    cases.check_view_vs_golden(r_my, g, "view_lego_")
    # a ray's early termination can flip on an fp16-level sigma difference; totals must be close
    a, b = int(g["view_lego_total_samples"]), int(r_my["total_samples"])
    assert abs(a - b) <= 0.01 * a + 8


def test_losses_match_reference(oracle):
    """NeRFLoss incl. the distortion term (reference losses.py) on the same compositing results"""
    from ngp_pl_b200.losses import NeRFLoss
    g = cases.golden("parity_render.npz")
    c = cases.loss_case(oracle)
    r = {k: torch.as_tensor(c[k]).cuda() for k in ("rgb", "opacity", "ws", "deltas", "ts", "rays_a")}
    r["ws"].requires_grad_(True)
    l_my = NeRFLoss(lambda_distortion=1e-3)(r, {"rgb": torch.as_tensor(c["target"]).cuda()})
    for k in ("rgb", "opacity", "distortion"):
        assert torch.allclose(l_my[k].float().cpu(), torch.as_tensor(g["loss_" + k]), rtol=1e-4, atol=3e-8), k
    # gradient of the distortion term w.r.t. ws
    g_my = torch.autograd.grad(l_my["distortion"].sum(), r["ws"])[0]
    assert torch.allclose(g_my.cpu(), torch.as_tensor(g["loss_dws"]), rtol=1e-4, atol=3e-8)


def test_mark_invisible_cells_matches_reference():
    from ngp_pl_b200 import synth
    from ngp_pl_b200.models.networks import NGP
    g = cases.golden("parity_render.npz")
    scale = 2.0
    mine = NGP(scale).cuda()
    G = 128
    coords = torch.stack(torch.meshgrid(*[torch.arange(G, dtype=torch.int32, device="cuda")] * 3, indexing="ij"), -1).reshape(-1, 3)
    mine.register_buffer("density_grid", torch.zeros(mine.cascades, G ** 3, device="cuda"))
    mine.register_buffer("grid_coords", coords)
    Kd = synth.intrinsics(W=200, H=150, fx=180.0)
    K = torch.tensor([[Kd["fx"], 0, Kd["cx"]], [0, Kd["fy"], Kd["cy"]], [0, 0, 1]], device="cuda")
    poses = torch.as_tensor(synth.camera_poses(6, radius=1.2)).cuda()
    mine.mark_invisible_cells(K, poses, (200, 150))
    frac = (mine.density_grid < 0).float().mean().item()
    assert cases.digest(mine.density_grid) == str(g["invisible_density"]), \
        "density_grid differs: %g of the cells invisible, reference %g" % (frac, float(g["invisible_fraction"]))
    # count_grid holds multiples of 1 / (6 cameras); compared as the camera counts
    count6 = torch.round(mine.count_grid * 6)
    assert torch.allclose(mine.count_grid, count6 / 6)
    assert cases.digest(count6.to(torch.uint8)) == str(g["invisible_count6"])
    assert 0 < frac < 1
