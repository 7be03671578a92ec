"""Generate tests/golden/parity_*.npz: what the REAL reference computes on the inputs of the GPU parity tests
(tests/test_vren_gpu.py, tests/test_render_gpu.py, tests/test_tcnn_modules_gpu.py), so that those tests compare
with the reference on any B200 without the reference installed. Needs oracle/_ref (oracle/build_ref.py) and a GPU:

    python tests/golden/make_golden_parity.py OUT_DIR

then copy OUT_DIR/parity_*.npz into tests/golden/. Inputs come from tests/cases.py (seeded).

  render_*   the reference's render() / NGP / NeRFLoss (its vren kernels, the tinycudann stand-in) on 2048 rays of each
             scene: per-ray counts, rgb / opacity / depth, and the parameter gradients -- rgb_net and the encoder MLP in
             full, the hash table as its largest magnitude plus 4096 seeded entries where the reference's gradient is
             non-zero (the full table is 48 MB); 100x100 test-time view: 2048 seeded rays of it and the sample total
  dropin_*   the same through the reference's unmodified Python bound to ngp_pl_b200.vren / ngp_pl_b200.tcnn
  ops        the reference's vren operators where the tests compare bit for bit (sha256 digests of the arrays, see
             cases.digest) or to a tolerance (the arrays)
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import cases  # noqa: E402
from oracle import oracle as O  # noqa: E402
from oracle import ref_env  # noqa: E402

N_TABLE_SAMPLES = 4096
N_VIEW_SAMPLES = 2048


def T(a, dtype=None):
    t = torch.as_tensor(np.ascontiguousarray(a)).cuda()
    return t.to(dtype) if dtype is not None else t


def f32(t):
    return t.detach().float().cpu().numpy()


def grads(model, prefix, out):
    p = dict(model.named_parameters())
    g = f32(p["rgb_net.params"].grad)
    out[prefix + "g_rgb_net"] = g
    g = f32(p["xyz_encoder.params"].grad)
    out[prefix + "g_xyz_scale"] = np.float32(np.abs(g).max())
    out[prefix + "g_xyz_mlp"] = g[:3072]
    nz = np.flatnonzero(g[3072:]) + 3072
    idx = np.sort(np.random.RandomState(0).choice(nz, min(N_TABLE_SAMPLES, nz.size), replace=False))
    out[prefix + "g_xyz_idx"] = idx.astype(np.int32)
    out[prefix + "g_xyz_val"] = g[idx]


def view_sample(res, prefix, out):
    n = res["rgb"].shape[0]
    idx = np.sort(np.random.RandomState(1).choice(n, N_VIEW_SAMPLES, replace=False))
    out[prefix + "idx"] = idx.astype(np.int32)
    for k in ("rgb", "opacity", "depth"):
        out[prefix + k] = f32(res[k])[idx]
    out[prefix + "total_samples"] = np.int64(int(res["total_samples"]))


def render_golden(ref, drop, out):
    from ngp_pl_b200 import synth
    for which in ("lego", "mip360"):
        scene = cases.scene_by_name(which)
        kw = {} if scene.exp_step_factor == 0 else {"exp_step_factor": scene.exp_step_factor}
        mine = cases.seeded_ngp(scene)
        sd = {k: v.clone() for k, v in mine.state_dict().items()}
        # test_render_gpu.py::test_train_render_matches_reference
        theirs = ref.NGP(scene.scale).cuda()
        theirs.load_state_dict(sd, strict=True)
        o, d = (T(a) for a in cases.rays_from_scene(scene, 2048, 31, extra_edge_cases=False))
        torch.manual_seed(123)
        r = ref.render(theirs, o, d, **kw)
        pre = "render_%s_" % which
        ra = r["rays_a"][torch.argsort(r["rays_a"][:, 0])]
        out[pre + "rm_samples"] = np.int64(int(r["rm_samples"]))
        out[pre + "counts"] = ra[:, 2].cpu().numpy().astype(np.int32)
        for k in ("rgb", "opacity", "depth"):
            out[pre + k] = f32(r[k])
        out[pre + "keys"] = np.array(sorted(r.keys()))
        theirs.zero_grad()
        l = ref.losses.NeRFLoss(lambda_distortion=0)(r, {"rgb": cases.render_target(o.shape[0])})
        sum(v.mean() for v in l.values()).backward()
        grads(theirs, pre, out)

        # test_tcnn_modules_gpu.py::test_unmodified_reference_python_runs_on_our_vren_and_tcnn
        theirs = drop.NGP(scene.scale).cuda()
        theirs.load_state_dict(sd, strict=True)
        o, d = (T(a) for a in cases.rays_from_scene(scene, 2048, 51, extra_edge_cases=False))
        torch.manual_seed(5)
        r = drop.render(theirs, o, d, **kw)
        pre = "dropin_%s_" % which
        out[pre + "rm_samples"] = np.int64(int(r["rm_samples"]))
        out[pre + "rays_a"] = cases.digest(r["rays_a"])
        out[pre + "ts"] = cases.digest(r["ts"])
        for k in ("rgb", "opacity", "depth"):
            out[pre + k] = f32(r[k])
        tgt = cases.render_target(o.shape[0])
        op = r["opacity"] + 1e-10
        theirs.zero_grad()
        (((r["rgb"] - tgt) ** 2).mean() + (1e-3 * (-op * torch.log(op))).mean()).backward()
        grads(theirs, pre, out)
        K = synth.intrinsics(W=80, H=60, fx=1111.11 / 10)
        pose = torch.as_tensor(synth.camera_poses(3, radius=1.5 if which == "lego" else 0.9)[1]).cuda()
        o2, d2 = synth.get_rays(synth.ray_directions(K, "cuda"), pose)
        with torch.no_grad():
            view_sample(drop.render(theirs, o2, d2, test_time=True, **kw), pre + "view_", out)

    # test_render_gpu.py::test_test_render_matches_reference
    scene = synth.lego_scene(0)
    theirs = ref.NGP(scene.scale).cuda()
    theirs.load_state_dict(cases.seeded_ngp(scene).state_dict(), strict=True)
    K = synth.intrinsics(W=100, H=100, fx=1111.11 / 8)
    o, d = synth.get_rays(synth.ray_directions(K, "cuda"), torch.as_tensor(synth.camera_poses(3)[2]).cuda())
    with torch.no_grad():
        view_sample(ref.render(theirs, o, d, test_time=True), "view_lego_", out)

    # test_render_gpu.py::test_losses_match_reference
    c = cases.loss_case(O)
    r = {k: T(c[k]) for k in ("rgb", "opacity", "ws", "deltas", "ts", "rays_a")}
    r["ws"].requires_grad_(True)
    l = ref.losses.NeRFLoss(lambda_distortion=1e-3)(r, {"rgb": T(c["target"])})
    for k in ("rgb", "opacity", "distortion"):
        out["loss_" + k] = f32(l[k])
    out["loss_dws"] = f32(torch.autograd.grad(l["distortion"].sum(), r["ws"])[0])

    # test_render_gpu.py::test_mark_invisible_cells_matches_reference
    scale, G = 2.0, 128
    m = ref.NGP(scale).cuda()
    coords = torch.stack(torch.meshgrid(*[torch.arange(G, dtype=torch.int32, device="cuda")] * 3, indexing="ij"), -1).reshape(-1, 3)
    m.register_buffer("density_grid", torch.zeros(m.cascades, G ** 3, device="cuda"))
    m.register_buffer("grid_coords", coords)
    Kd = synth.intrinsics(W=200, H=150, fx=180.0)
    Km = torch.tensor([[Kd["fx"], 0, Kd["cx"]], [0, Kd["fy"], Kd["cy"]], [0, 0, 1]], device="cuda")
    m.mark_invisible_cells(Km, torch.as_tensor(synth.camera_poses(6, radius=1.2)).cuda(), (200, 150))
    out["invisible_density"] = cases.digest(m.density_grid)
    out["invisible_count6"] = cases.digest(torch.round(m.count_grid * 6).to(torch.uint8))
    out["invisible_fraction"] = np.float64((m.density_grid < 0).double().mean().item())


def ops_golden(vren, out):
    from ngp_pl_b200 import synth
    # test_vren_gpu.py::test_march_test_rounds
    for name in cases.MARCH_CASES:
        c = cases.march_case(name)
        o, d, bits = T(c["o"]), T(c["d"]), T(c["bits"])
        hits = T(cases.hits_for(c, O).copy())
        alive = torch.arange(o.shape[0], device="cuda")
        for ns in (1, 2, 4, 64):
            r = vren.raymarching_test(o, d, hits, alive, bits, c["cascades"], float(c["scale"]), float(c["esf"]), 128, 1024, ns)
            for t, nm in zip(r[:4], ["xyzs", "dirs", "deltas", "ts"]):
                out["test_%s_%d_%s" % (name, ns, nm)] = cases.digest(t)
            out["test_%s_%d_neff" % (name, ns)] = cases.digest(r[4].long())
            out["test_%s_%d_hits" % (name, ns)] = cases.digest(hits)

    # test_vren_gpu.py::test_march_large_vs_reference
    for which, esf, n_rays in cases.LARGE_MARCH:
        pre = "large_%s_" % which
        scene = cases.scene_by_name(which)
        bits = T(synth.pack_bits(synth.occupancy_grid(scene)))
        o, d = (T(a) for a in cases.rays_from_scene(scene, n_rays, 77))
        center = torch.zeros(1, 3, device="cuda")
        half = torch.full((1, 3), scene.scale, device="cuda")
        _, hits_t, _ = vren.ray_aabb_intersect(o, d, center, half, 1)
        out[pre + "hits"] = cases.digest(hits_t)
        t0 = hits_t[:, 0, 0]
        hits_t[:, 0, 0] = torch.where((t0 >= 0) & (t0 < 0.01), torch.full_like(t0, 0.01), t0)
        hits = hits_t[:, 0].contiguous()
        noise = torch.rand(n_rays, device="cuda", generator=torch.Generator("cuda").manual_seed(5))
        ra, xyz, _, dl, ts, cnt = vren.raymarching_train(o, d, hits, bits, scene.cascades, scene.scale, esf, noise, 128, 1024)
        tot = int(cnt[0])
        ra = ra[torch.argsort(ra[:, 0])]
        start = torch.cumsum(ra[:, 2], 0) - ra[:, 2]
        seg = torch.repeat_interleave(torch.arange(n_rays, device="cuda"), ra[:, 2])
        src = ra[:, 1][seg] + torch.arange(tot, device="cuda") - start[seg]
        out[pre + "total"] = np.int64(tot)
        out[pre + "counts"] = cases.digest(ra[:, 2].long())
        for t, nm in ((ts, "ts"), (dl, "deltas"), (xyz, "xyzs")):
            out[pre + nm] = cases.digest(t[src])

    # test_vren_gpu.py::test_composite_test_fw
    c = cases.composite_test_case()
    alive, op, dp, rgb = T(c["alive"]), T(c["opacity"]), T(c["depth"]), T(c["rgb"])
    vren.composite_test_fw(T(c["sigmas"]), T(c["rgbs"]), T(c["deltas"]), T(c["ts"]), torch.zeros(200, 2, device="cuda"), alive, 1e-2,
                           T(c["neff"]), op, dp, rgb)
    out["ctest_alive"], out["ctest_opacity"], out["ctest_rgb"] = alive.cpu().numpy(), f32(op), f32(rgb)

    # test_vren_gpu.py::test_distortion_loss
    c = cases.composite_case(seed=9)
    _, _, _, _, ws_np = O.composite_train_fw(c["sigmas"], c["rgbs"], c["deltas"], c["ts"], c["rays_a"], 1e-4)
    ws, dl, ts, ra = T(ws_np), T(c["deltas"]), T(c["ts"]), T(c["rays_a"])
    loss, wi, wti = vren.distortion_loss_fw(ws, dl, ts, ra)
    dL = np.random.RandomState(8).normal(size=ra.shape[0]).astype(np.float32)
    out["dist_loss"], out["dist_dws"] = f32(loss), f32(vren.distortion_loss_bw(T(dL), wi, wti, ws, dl, ts, ra))

    # test_vren_gpu.py::test_packbits_morton (the same draws from the same RandomState)
    rng = np.random.RandomState(21)
    for dtype in (torch.float32, torch.float16, torch.float64):
        g = T(rng.normal(0, 1, 4096 * 8).astype(np.float32)).to(dtype)
        bf = torch.zeros(4096, dtype=torch.uint8, device="cuda")
        vren.packbits(g, 0.25, bf)
        out["packbits_" + str(dtype).split(".")[1]] = cases.digest(bf)
    rng.normal(0, 1, 1001 * 8)
    rng.randint(0, 1024, (5000, 3))
    c128 = T(rng.randint(0, 128, (5000, 3)).astype(np.int32))
    m = vren.morton3D(c128)
    out["morton128"] = cases.digest(m.long())
    out["morton128_invert"] = cases.digest(vren.morton3D_invert(m).long())


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    O.build()
    ref = ref_env.load_reference()
    drop = ref_env.load_reference(drop_in=True)
    out = {}
    ops_golden(ref.vren, out)
    np.savez_compressed(os.path.join(out_dir, "parity_ops.npz"), **out)
    out = {}
    render_golden(ref, drop, out)
    np.savez_compressed(os.path.join(out_dir, "parity_render.npz"), **out)
    print("golden written to", out_dir)


if __name__ == "__main__":
    main(sys.argv[1])
