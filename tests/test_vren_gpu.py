"""GPU parity of the twelve vren operators (through the C ABI) against
  (1) the CPU oracle (oracle/ngp_oracle.c) on the same seeded inputs, and
  (2) the REAL reference kernels on the same inputs, as stored in tests/golden/ (march_*.npz, composite.npz,
      parity_ops.npz; arrays, or sha256 digests where the comparison is bit for bit).
Marcher: per-ray sample counts and the t / dt / xyz sequences are BIT-EXACT.
Compositing / distortion: 1e-4 relative (the reference uses __expf and serial fp32 sums).
"""
import numpy as np
import pytest
import torch

import cases

pytestmark = pytest.mark.gpu

RTOL = 1e-4


def T(a, dtype=None):
    t = torch.as_tensor(np.ascontiguousarray(a)).cuda()
    return t.to(dtype) if dtype is not None else t


def rel_close(a, b, rtol=RTOL, atol=1e-6, what=""):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    err = np.abs(a - b)
    lim = atol + rtol * np.maximum(np.abs(a), np.abs(b))
    bad = err > lim
    assert not bad.any(), "%s: %d/%d outside rtol=%g; worst abs err %g at %s (%g vs %g)" % (
        what, bad.sum(), bad.size, rtol, err.max(), np.unravel_index(err.argmax(), err.shape),
        a.flat[err.argmax()], b.flat[err.argmax()])


def bits_equal(a, b, what=""):
    a = np.ascontiguousarray(a, np.float32).view(np.uint32)
    b = np.ascontiguousarray(b, np.float32).view(np.uint32)
    assert a.shape == b.shape, "%s: shape %s vs %s" % (what, a.shape, b.shape)
    bad = a != b
    assert not bad.any(), "%s: %d/%d elements differ bitwise, first at %s" % (
        what, bad.sum(), bad.size, np.argwhere(bad)[0] if bad.any() else None)


def my_aabb(c):
    from ngp_pl_b200 import vren
    center = torch.zeros(1, 3, device="cuda")
    half = torch.full((1, 3), float(c["scale"]), device="cuda")
    return vren.ray_aabb_intersect(T(c["o"]), T(c["d"]), center, half, 1)


def near_clamp(hits_t):
    t0 = hits_t[:, 0, 0]
    hits_t[:, 0, 0] = torch.where((t0 >= 0) & (t0 < 0.01), torch.full_like(t0, 0.01), t0)
    return hits_t[:, 0].contiguous()


@pytest.mark.parametrize("name", cases.MARCH_CASES)
def test_aabb_and_march_train_vs_oracle(name, oracle):
    from ngp_pl_b200 import vren
    c = cases.march_case(name)
    cnt, hits_t, idx = my_aabb(c)
    hits_o = cases.hits_for(c, oracle)
    hits = near_clamp(hits_t)
    bits_equal(hits.cpu().numpy(), hits_o, "hits_t")
    assert ((hits_o[:, 1] > 0) == (cnt.cpu().numpy() == 1)).all()

    rays_a, xyzs, dirs, deltas, ts, counter = vren.raymarching_train(
        T(c["o"]), T(c["d"]), hits, T(c["bits"]), c["cascades"], float(c["scale"]), float(c["esf"]), T(c["noise"]), 128, 1024)
    ra_o, xyz_o, dir_o, dl_o, ts_o = oracle.march_train(c["o"], c["d"], hits_o, c["bits"], c["cascades"], c["scale"],
                                                        c["esf"], c["noise"], 128, 1024)
    total = int(counter[0])
    assert int(counter[1]) == c["o"].shape[0]
    assert (rays_a.cpu().numpy() == ra_o).all(), "rays_a (ray_idx,start,N) differs from the oracle"
    assert total == ra_o[:, 2].sum()
    bits_equal(ts[:total].cpu().numpy(), ts_o, "ts")
    bits_equal(deltas[:total].cpu().numpy(), dl_o, "deltas")
    bits_equal(xyzs[:total].cpu().numpy(), xyz_o, "xyzs")
    bits_equal(dirs[:total].cpu().numpy(), dir_o, "dirs")
    if name == "full_scale2":
        assert ra_o[:, 2].max() == 1024 and (ra_o[:, 2] == 1024).sum() >= 4  # max_samples saturation is exercised


@pytest.mark.parametrize("name", cases.MARCH_CASES)
def test_march_train_vs_reference_kernels(name):
    from ngp_pl_b200 import vren
    g = cases.golden("march_%s.npz" % name)
    c = cases.march_case(name)
    o, d, bits, noise = T(c["o"]), T(c["d"]), T(c["bits"]), T(c["noise"])
    center = torch.zeros(1, 3, device="cuda")
    half = torch.full((1, 3), float(c["scale"]), device="cuda")
    cnt_m, hits_m, _ = vren.ray_aabb_intersect(o, d, center, half, 1)
    bits_equal(hits_m.cpu().numpy(), g["hits_raw"], "ray_aabb_intersect hits_t")
    assert (cnt_m.cpu().numpy() == g["hit_cnt"]).all()
    hits = near_clamp(hits_m)
    args = (o, d, hits, bits, c["cascades"], float(c["scale"]), float(c["esf"]), noise, 128, 1024)
    ra_m, xyz_m, dir_m, dl_m, ts_m, cnt_m2 = vren.raymarching_train(*args)
    tot = int(cnt_m2[0])
    assert tot == int(g["total"])
    assert (ra_m[:, 2].cpu().numpy() == g["counts"]).all(), "per-ray sample counts differ from the reference kernel"
    bits_equal(ts_m[:tot].cpu().numpy(), g["ts"], "ts vs reference")
    bits_equal(dl_m[:tot].cpu().numpy(), g["deltas"], "deltas vs reference")
    bits_equal(xyz_m[:tot].cpu().numpy(), g["xyzs"], "xyzs vs reference")


@pytest.mark.parametrize("name", cases.MARCH_CASES)
def test_march_test_rounds(name, oracle):
    from ngp_pl_b200 import vren
    g = cases.golden("parity_ops.npz")
    c = cases.march_case(name)
    o, d, bits = T(c["o"]), T(c["d"]), T(c["bits"])
    hits_np = cases.hits_for(c, oracle).copy()
    hits_m = T(hits_np)
    n = o.shape[0]
    alive = torch.arange(n, device="cuda")
    for ns in (1, 2, 4, 64):
        out_m = vren.raymarching_test(o, d, hits_m, alive, bits, c["cascades"], float(c["scale"]), float(c["esf"]), 128, 1024, ns)
        out_o = oracle.march_test(c["o"], c["d"], hits_np, np.arange(n), c["bits"], c["cascades"], c["scale"], c["esf"],
                                  128, 1024, ns)
        for a, b, nm in zip(out_m[:4], out_o[:4], ["xyzs", "dirs", "deltas", "ts"]):
            bits_equal(a.cpu().numpy(), b, "raymarching_test %s (N_samples=%d)" % (nm, ns))
        assert (out_m[4].cpu().numpy() == out_o[4]).all()
        bits_equal(hits_m.cpu().numpy(), hits_np, "hits_t after round")
        key = "test_%s_%d_" % (name, ns)
        for a, nm in zip(out_m[:4], ["xyzs", "dirs", "deltas", "ts"]):
            assert cases.digest(a) == str(g[key + nm]), "raymarching_test %s (N_samples=%d) vs reference" % (nm, ns)
        assert cases.digest(out_m[4].long()) == str(g[key + "neff"]), "N_eff_samples vs reference"
        assert cases.digest(hits_m) == str(g[key + "hits"]), "hits_t vs reference"


def test_march_large_vs_reference():
    """bit-exactness over many rays (size-independent check at the bench's ray count and beyond)"""
    from ngp_pl_b200 import synth, vren
    g = cases.golden("parity_ops.npz")
    for which, esf, n_rays in cases.LARGE_MARCH:
        pre = "large_%s_" % which
        scene = cases.scene_by_name(which)
        bits = T(synth.pack_bits(synth.occupancy_grid(scene)))
        o_np, d_np = cases.rays_from_scene(scene, n_rays, 77)
        o, d = T(o_np), T(d_np)
        center = torch.zeros(1, 3, device="cuda")
        half = torch.full((1, 3), scene.scale, device="cuda")
        _, hits_m, _ = vren.ray_aabb_intersect(o, d, center, half, 1)
        assert cases.digest(hits_m) == str(g[pre + "hits"]), "%s: ray_aabb_intersect vs reference" % which
        hits = near_clamp(hits_m)
        noise = torch.rand(n_rays, device="cuda", generator=torch.Generator("cuda").manual_seed(5))
        args = (o, d, hits, bits, scene.cascades, scene.scale, esf, noise, 128, 1024)
        ra_m, xyz_m, _, dl_m, ts_m, cnt_m = vren.raymarching_train(*args)
        tot = int(cnt_m[0])
        assert tot == int(g[pre + "total"]) and tot > 0
        assert cases.digest(ra_m[:, 2].long()) == str(g[pre + "counts"]), "%s: per-ray sample counts vs reference" % which
        # the reference's samples are stored gathered into ray order
        for t, nm in ((ts_m, "ts"), (dl_m, "deltas"), (xyz_m, "xyzs")):
            assert cases.digest(t[:tot]) == str(g[pre + nm]), "%s: %s vs reference" % (which, nm)


def test_composite_train_fw_bw(oracle):
    from ngp_pl_b200 import vren
    c = cases.composite_case()
    sig, rgbs, dl, ts, ra = T(c["sigmas"]), T(c["rgbs"]), T(c["deltas"]), T(c["ts"]), T(c["rays_a"])
    thr = float(c["T_thr"])
    total, opacity, depth, rgb, ws = vren.composite_train_fw(sig, rgbs, dl, ts, ra, thr)
    o_total, o_op, o_dp, o_rgb, o_ws = oracle.composite_train_fw(c["sigmas"], c["rgbs"], c["deltas"], c["ts"], c["rays_a"], thr)
    assert (total.cpu().numpy() == o_total).all()
    rel_close(opacity.cpu().numpy(), o_op, what="opacity")
    rel_close(depth.cpu().numpy(), o_dp, what="depth")
    rel_close(rgb.cpu().numpy(), o_rgb, what="rgb")
    rel_close(ws.cpu().numpy(), o_ws, atol=2e-6, what="ws")
    dsig, drgbs = vren.composite_train_bw(T(c["dO"]), T(c["dD"]), T(c["dC"]), T(c["dws"]), sig, rgbs, ws, dl, ts, ra,
                                          opacity, depth, rgb, thr)
    o_dsig, o_drgbs = oracle.composite_train_bw(c["dO"], c["dD"], c["dC"], c["dws"], c["sigmas"], c["rgbs"], o_ws, c["deltas"],
                                                c["ts"], c["rays_a"], o_op, o_dp, o_rgb, thr)
    rel_close(drgbs.cpu().numpy(), o_drgbs, atol=1e-5, what="dL_drgbs")
    # dL_dsigmas is a difference of O(1) terms scaled by delta: absolute floor = 1e-4 * delta * |terms|
    rel_close(dsig.cpu().numpy(), o_dsig, atol=1e-5, what="dL_dsigmas")
    g = cases.golden("composite.npz")
    assert (total.cpu().numpy() == g["total"]).all()
    rel_close(opacity.cpu().numpy(), g["opacity"], what="opacity vs reference")
    rel_close(rgb.cpu().numpy(), g["rgb"], what="rgb vs reference")
    rel_close(depth.cpu().numpy(), g["depth"], what="depth vs reference")
    rel_close(ws.cpu().numpy(), g["ws"], atol=2e-6, what="ws vs reference")
    rel_close(drgbs.cpu().numpy(), g["drgbs"], atol=1e-5, what="dL_drgbs vs reference")
    rel_close(dsig.cpu().numpy(), g["dsig"], atol=1e-5, what="dL_dsigmas vs reference")


def test_composite_test_fw(oracle):
    from ngp_pl_b200 import vren
    c = cases.composite_test_case()
    alive_np, sig, rgbs, dl, ts, neff = c["alive"], c["sigmas"], c["rgbs"], c["deltas"], c["ts"], c["neff"]
    op0, dp0, rgb0 = c["opacity"], c["depth"], c["rgb"]
    n_rays = op0.shape[0]
    alive_m, op_m, dp_m, rgb_m = T(alive_np), T(op0), T(dp0), T(rgb0)
    hits = torch.zeros(n_rays, 2, device="cuda")
    vren.composite_test_fw(T(sig), T(rgbs), T(dl), T(ts), hits, alive_m, 1e-2, T(neff), op_m, dp_m, rgb_m)
    alive_o, op_o, dp_o, rgb_o = alive_np.copy(), op0.copy(), dp0.copy(), rgb0.copy()
    oracle.composite_test_fw(sig, rgbs, dl, ts, alive_o, 1e-2, neff, op_o, dp_o, rgb_o)
    assert (alive_m.cpu().numpy() == alive_o).all()
    rel_close(op_m.cpu().numpy(), op_o, what="opacity")
    rel_close(dp_m.cpu().numpy(), dp_o, what="depth")
    rel_close(rgb_m.cpu().numpy(), rgb_o, what="rgb")
    g = cases.golden("parity_ops.npz")
    assert (alive_m.cpu().numpy() == g["ctest_alive"]).all()
    rel_close(op_m.cpu().numpy(), g["ctest_opacity"], what="opacity vs reference")
    rel_close(rgb_m.cpu().numpy(), g["ctest_rgb"], what="rgb vs reference")


def test_distortion_loss(oracle):
    from ngp_pl_b200 import vren
    c = cases.composite_case(seed=9)
    _, _, _, _, ws_np = oracle.composite_train_fw(c["sigmas"], c["rgbs"], c["deltas"], c["ts"], c["rays_a"], 1e-4)
    ws, dl, ts, ra = T(ws_np), T(c["deltas"]), T(c["ts"]), T(c["rays_a"])
    loss, wi, wti = vren.distortion_loss_fw(ws, dl, ts, ra)
    o_loss, o_wi, o_wti = oracle.distortion_fw(ws_np, c["deltas"], c["ts"], c["rays_a"])
    rel_close(wi.cpu().numpy(), o_wi, atol=1e-7, what="ws_inclusive_scan")
    rel_close(wti.cpu().numpy(), o_wti, atol=1e-7, what="wts_inclusive_scan")
    # the per-ray loss is a difference of O(1) prefix products: absolute, not relative, accuracy
    rel_close(loss.cpu().numpy(), o_loss, atol=3e-5, what="distortion loss")
    dL = np.random.RandomState(8).normal(size=ra.shape[0]).astype(np.float32)
    dws = vren.distortion_loss_bw(T(dL), wi, wti, ws, dl, ts, ra)
    o_dws = oracle.distortion_bw(dL, o_wi, o_wti, ws_np, c["deltas"], c["ts"], c["rays_a"])
    rel_close(dws.cpu().numpy(), o_dws, atol=3e-5, what="dL_dws")
    g = cases.golden("parity_ops.npz")
    rel_close(loss.cpu().numpy(), g["dist_loss"], atol=3e-5, what="distortion loss vs reference")
    rel_close(dws.cpu().numpy(), g["dist_dws"], atol=3e-5, what="dL_dws vs reference")


def test_packbits_morton(oracle):
    from ngp_pl_b200 import vren
    gold = cases.golden("parity_ops.npz")
    rng = np.random.RandomState(21)
    for dtype in (torch.float32, torch.float16, torch.float64):
        grid = rng.normal(0, 1, 4096 * 8).astype(np.float32)
        g = T(grid).to(dtype)
        bf = torch.zeros(4096, dtype=torch.uint8, device="cuda")
        vren.packbits(g, 0.25, bf)
        want = oracle.packbits(g.float().cpu().numpy(), 0.25) if dtype != torch.float64 else oracle.packbits(grid, 0.25)
        assert (bf.cpu().numpy() == want).all()
        assert cases.digest(bf) == str(gold["packbits_" + str(dtype).split(".")[1]]), "packbits %s vs reference" % dtype
    # odd size (not a multiple of 4 bytes) takes the byte path
    grid = rng.normal(0, 1, 1001 * 8).astype(np.float32)
    bf = torch.zeros(1001, dtype=torch.uint8, device="cuda")
    vren.packbits(T(grid), -0.1, bf)
    assert (bf.cpu().numpy() == oracle.packbits(grid, -0.1)).all()

    coords = rng.randint(0, 1024, (5000, 3)).astype(np.int32)
    coords[:3] = [[0, 0, 0], [1023, 1023, 1023], [127, 0, 64]]
    m = vren.morton3D(T(coords))
    assert (m.cpu().numpy() == oracle.morton3D(coords)).all()
    inv = vren.morton3D_invert(m)
    assert (inv.cpu().numpy() == coords).all()
    c128 = T(rng.randint(0, 128, (5000, 3)).astype(np.int32))
    m = vren.morton3D(c128)
    assert cases.digest(m.long()) == str(gold["morton128"]), "morton3D vs reference"
    assert cases.digest(vren.morton3D_invert(m).long()) == str(gold["morton128_invert"]), "morton3D_invert vs reference"


def test_empty_and_error_paths():
    from ngp_pl_b200 import vren
    e3 = torch.zeros(0, 3, device="cuda")
    cnt, hits, idx = vren.ray_aabb_intersect(e3, e3, torch.zeros(1, 3, device="cuda"), torch.ones(1, 3, device="cuda"), 1)
    assert hits.shape == (0, 1, 2)
    out = vren.raymarching_train(e3, e3, torch.zeros(0, 2, device="cuda"), torch.zeros(128 ** 3 // 8, dtype=torch.uint8, device="cuda"),
                                 1, 0.5, 0.0, torch.zeros(0, device="cuda"), 128, 1024)
    assert int(out[5][0]) == 0
    with pytest.raises(RuntimeError):
        vren.morton3D(torch.zeros(4, 3, dtype=torch.int32))  # CPU tensor -> RuntimeError, like TORCH_CHECK(is_cuda)
    with pytest.raises(RuntimeError):
        vren.morton3D(torch.zeros(4, 6, dtype=torch.int32, device="cuda")[:, ::2])  # non-contiguous
