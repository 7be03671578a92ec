"""The tinycudann-shaped modules called one by one (ngp_pl_b200/tcnn.py), and the strongest drop-in check:
the reference's UNMODIFIED models/{networks,rendering,custom_functions}.py running on
    vren        = ngp_pl_b200.vren
    tinycudann  = ngp_pl_b200.tcnn
compared with this repo's fused NGP / render on identical rays, weights and jitter.
"""
import numpy as np
import pytest
import torch

import cases

pytestmark = pytest.mark.gpu


def test_sh_encoding_matches_oracle(oracle):
    from ngp_pl_b200 import tcnn
    enc = tcnn.Encoding(3, {"otype": "SphericalHarmonics", "degree": 4}).cuda()
    d = torch.randn(5000, 3, device="cuda")
    d = d / d.norm(dim=1, keepdim=True)
    out = enc((d + 1) / 2)
    assert out.dtype == torch.float16 and out.shape == (5000, 16)
    want = oracle.torch_sh4(((d + 1) / 2 * 2 - 1).cpu()).half()
    assert (out.cpu().float() - want.float()).abs().max().item() < 2e-3


def test_rgb_network_forward_backward(oracle):
    from ngp_pl_b200 import tcnn
    net = tcnn.Network(32, 3, {"otype": "FullyFusedMLP", "activation": "ReLU", "output_activation": "Sigmoid",
                               "n_neurons": 64, "n_hidden_layers": 2}).cuda()
    n = 3001
    x = (torch.randn(n, 32, device="cuda") * 0.5).half().requires_grad_(True)
    w = torch.randn(n, 3, device="cuda") * 1e-3
    out = net(x)
    assert out.dtype == torch.float16 and out.shape == (n, 3)
    (out.float() * w).sum().backward()
    # fp32 torch restatement with the same rounding points
    p = net.params.detach().cpu().clone().requires_grad_(True)
    xr = x.detach().cpu().float().requires_grad_(True)
    rt = oracle._rt
    ph = rt(p)
    r1 = rt(torch.relu(xr @ ph[:2048].view(64, 32).t()))
    r2 = rt(torch.relu(r1 @ ph[2048:6144].view(64, 64).t()))
    o = rt(torch.sigmoid((r2 @ ph[6144:].view(16, 64).t())[:, :3]))
    (o * w.cpu()).sum().backward()
    assert (out.cpu().float() - o.detach()).abs().max().item() < 4e-3
    gs = p.grad.abs().max().item()
    assert (net.params.grad.cpu() - p.grad).abs().max().item() < 0.03 * gs
    xs = xr.grad.abs().max().item()
    assert (x.grad.cpu().float() - xr.grad).abs().max().item() < 0.03 * xs


def test_encoder_network_forward_backward(oracle):
    from ngp_pl_b200 import tcnn
    b = float(np.exp(np.log(2048 * 0.5 / 16) / 15))
    m = tcnn.NetworkWithInputEncoding(
        3, 16, {"otype": "Grid", "type": "Hash", "n_levels": 16, "n_features_per_level": 2, "log2_hashmap_size": 19,
                "base_resolution": 16, "per_level_scale": b, "interpolation": "Linear"},
        {"otype": "FullyFusedMLP", "activation": "ReLU", "output_activation": "None", "n_neurons": 64, "n_hidden_layers": 1}).cuda()
    with torch.no_grad():
        m.params[3072:].uniform_(-0.5, 0.5)
    n = 2000 + 5
    x01 = torch.rand(n, 3, device="cuda")
    w = torch.randn(n, 16, device="cuda") * 1e-3
    h = m(x01)
    assert h.dtype == torch.float16 and h.shape == (n, 16)
    (h.float() * w).sum().backward()
    p = m.params.detach().cpu().clone().requires_grad_(True)
    meta, _ = oracle.grid_meta(16, 19, 16, float(np.float32(b)))
    ph = oracle._rt(p)
    feat = oracle.torch_grid_encode(meta, ph[3072:].view(-1, 2), x01.cpu())
    hid = oracle._rt(torch.relu(feat @ ph[:2048].view(64, 32).t()))
    ho = oracle._rt(hid @ ph[2048:3072].view(16, 64).t())
    (ho * w.cpu()).sum().backward()
    assert (h.cpu().float() - ho.detach()).abs().max().item() < 0.01 * max(1.0, ho.abs().max().item())
    for lo, hi, name in ((0, 2048, "W1"), (2048, 3072, "W2"), (3072, p.numel(), "table")):
        s = p.grad[lo:hi].abs().max().item()
        e = (m.params.grad.cpu()[lo:hi] - p.grad[lo:hi]).abs().max().item()
        assert e < 0.03 * s, "%s: %g vs %g" % (name, e, s)


@pytest.mark.parametrize("which", ["lego", "mip360"])
def test_unmodified_reference_python_runs_on_our_vren_and_tcnn(which):
    """the reference's own NGP / render / autograd Functions, bound to OUR vren and OUR tcnn (stored in
    tests/golden/parity_render.npz by tests/golden/make_golden_parity.py)"""
    from ngp_pl_b200 import synth
    from ngp_pl_b200.models.rendering import render
    g = cases.golden("parity_render.npz")
    pre = "dropin_%s_" % which
    scene = cases.scene_by_name(which)
    mine = cases.seeded_ngp(scene)
    o_np, d_np = cases.rays_from_scene(scene, 2048, 51, extra_edge_cases=False)
    o, d = torch.as_tensor(o_np).cuda(), torch.as_tensor(d_np).cuda()
    kw = {} if scene.exp_step_factor == 0 else {"exp_step_factor": scene.exp_step_factor}
    torch.manual_seed(5)
    r_my = render(mine, o, d, **kw)
    assert int(g[pre + "rm_samples"]) == int(r_my["rm_samples"]) > 0
    assert cases.digest(r_my["rays_a"]) == str(g[pre + "rays_a"])
    assert cases.digest(r_my["ts"]) == str(g[pre + "ts"])
    for k in ("rgb", "opacity", "depth"):
        ref_k = g[pre + k]
        err = np.abs(ref_k - r_my[k].detach().float().cpu().numpy()).max()
        assert err < 3e-3 * max(1.0, np.abs(ref_k).max()), "%s differs by %g" % (k, err)
    tgt = cases.render_target(o.shape[0])
    op = r_my["opacity"] + 1e-10
    mine.zero_grad()
    (((r_my["rgb"] - tgt) ** 2).mean() + (1e-3 * (-op * torch.log(op))).mean()).backward()
    cases.check_grads_vs_golden(mine, g, pre, 0.05)
    # test-time render through the reference's host loop on our operators vs our device-side wavefront
    K = synth.intrinsics(W=80, H=60, fx=1111.11 / 10)
    dirs = synth.ray_directions(K, "cuda")
    pose = torch.as_tensor(synth.camera_poses(3, radius=1.5 if which == "lego" else 0.9)[1]).cuda()
    o2, d2 = synth.get_rays(dirs, pose)
    cases.check_view_vs_golden(render(mine, o2, d2, test_time=True, **kw), g, pre + "view_")
