"""Deterministic parity cases shared by tests/golden/make_golden.py (runs the REAL reference on a B200),
the CPU-oracle tests and the GPU parity tests. numpy RandomState only, so every host builds the
same inputs."""
import hashlib
import os

import numpy as np
import torch

from ngp_pl_b200 import synth

NEAR = np.float32(0.01)
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden(name):
    """a stored result of the reference (tests/golden/make_golden*.py)"""
    return np.load(os.path.join(GOLDEN, name))


def rays_from_scene(scene, n_rays, seed, extra_edge_cases=True):
    rng = np.random.RandomState(seed)
    K = synth.intrinsics()
    dirs = synth.ray_directions(K)
    radius = 1.5 if scene.scale <= 0.5 else 0.9
    poses = torch.as_tensor(synth.camera_poses(8, radius=radius, seed=seed))
    img = rng.randint(0, 8, n_rays)
    pix = rng.randint(0, dirs.shape[0], n_rays)
    o, d = synth.get_rays(dirs[torch.as_tensor(pix)], poses[torch.as_tensor(img)])
    o, d = o.numpy().copy(), d.numpy().copy()
    if extra_edge_cases and n_rays >= 16:
        s = scene.scale
        # axis-parallel rays (1/0 = inf), a ray starting inside the box, a ray pointing away, a grazing ray
        o[0], d[0] = [-2 * s - 1, 0.01, 0.02], [1, 0, 0]
        o[1], d[1] = [0.03, -2 * s - 1, -0.1 * s], [0, 1, 0]
        o[2], d[2] = [0.0, 0.1 * s, 2 * s + 1], [0, 0, -1]
        o[3], d[3] = [0.01, 0.02, 0.03], [0.3, -0.5, 0.8]
        o[4], d[4] = [3 * s, 3 * s, 3 * s], [1, 1, 1]
        o[5], d[5] = [-2 * s, s * 0.999999, 0.0], [1, 0, 1e-4]
        o[6], d[6] = [0.0, 0.0, 0.005], [1, 1, 0]  # starts inside, t0 < NEAR
    return o.astype(np.float32), d.astype(np.float32)


def march_case(name):
    """-> dict(scene, bits, o, d, noise, cascades, scale, esf, grid_size, max_samples)"""
    if name == "lego":
        sc = synth.lego_scene(0)
        bits = synth.pack_bits(synth.occupancy_grid(sc))
        o, d = rays_from_scene(sc, 256, 11)
        esf = 0.0
    elif name == "lego_half_random":
        # what the grid looks like during warm-up: ~half of the cells set, no structure
        sc = synth.lego_scene(0)
        rng = np.random.RandomState(5)
        bits = rng.randint(0, 256, 128 ** 3 // 8).astype(np.uint8)
        o, d = rays_from_scene(sc, 64, 12)
        esf = 0.0
    elif name == "full":
        sc = synth.lego_scene(0)
        bits = np.full(128 ** 3 // 8, 255, np.uint8)  # saturates max_samples on the diagonal
        o, d = rays_from_scene(sc, 32, 13)
        esf = 0.0
    elif name == "full_scale2":
        # scale 2 => 3 cascades, chords several units long at the minimum step: saturates max_samples = 1024
        sc = synth.Scene(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32), 2.0, 0.0)
        bits = np.full(sc.cascades * 128 ** 3 // 8, 255, np.uint8)
        o, d = rays_from_scene(sc, 32, 15)
        esf = 0.0
    elif name == "mip360":
        sc = synth.mip360_scene(0)
        bits = synth.pack_bits(synth.occupancy_grid(sc))
        o, d = rays_from_scene(sc, 128, 14)
        esf = 1.0 / 256
    else:
        raise KeyError(name)
    rng = np.random.RandomState(99)
    noise = rng.rand(o.shape[0]).astype(np.float32)
    return dict(scene=sc, bits=bits, o=o, d=d, noise=noise, cascades=sc.cascades, scale=np.float32(sc.scale),
                esf=np.float32(esf), grid_size=128, max_samples=1024)


MARCH_CASES = ["lego", "lego_half_random", "full", "full_scale2", "mip360"]

# (scene, exp_step_factor, rays): bit-exactness of the marcher at the bench's ray count and beyond
LARGE_MARCH = [("lego", 0.0, 1 << 18), ("mip360", 1.0 / 256, 1 << 16)]


def composite_case(seed=3, n_rays=96, max_n=300):
    """ragged random samples: sigmas, rgbs, deltas, ts, rays_a (+ upstream gradients)"""
    rng = np.random.RandomState(seed)
    counts = rng.randint(0, max_n, n_rays)
    counts[:4] = [0, 1, 32, 33]
    counts[4] = 700
    start = np.concatenate([[0], np.cumsum(counts)[:-1]])
    n = int(counts.sum())
    rays_a = np.stack([rng.permutation(n_rays), start, counts], 1).astype(np.int64)
    sig = np.exp(rng.normal(0, 2.5, n)).astype(np.float32)
    sig[rng.rand(n) < 0.3] *= 1e-3
    rgbs = rng.rand(n, 3).astype(np.float32)
    deltas = np.full(n, 1.73205080757 / 1024, np.float32) * rng.uniform(1, 8, n).astype(np.float32)
    ts = np.zeros(n, np.float32)
    for s, c in zip(start, counts):
        ts[s:s + c] = 0.3 + np.cumsum(deltas[s:s + c])
    g = dict(dO=rng.normal(size=n_rays).astype(np.float32), dD=rng.normal(size=n_rays).astype(np.float32),
             dC=rng.normal(size=(n_rays, 3)).astype(np.float32), dws=rng.normal(size=n).astype(np.float32))
    return dict(sigmas=sig, rgbs=rgbs, deltas=deltas, ts=ts, rays_a=rays_a, T_thr=np.float32(1e-4), **g)


def hits_for(case, oracle):
    return oracle.ray_aabb(case["o"], case["d"], np.zeros(3, np.float32), np.full(3, case["scale"], np.float32), NEAR)


def digest(a):
    """sha256 of an array's dtype, shape and bytes: a bit-exact comparison against a stored result too large to keep"""
    a = np.ascontiguousarray(a.detach().cpu().numpy() if torch.is_tensor(a) else a)
    h = hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return h.hexdigest()


def seeded_ngp(scene):
    """ngp_pl_b200's NGP on cuda with seeded weights (hash table ~U(-0.3, 0.3)) and the scene's occupancy bitfield"""
    from ngp_pl_b200.models.networks import NGP
    m = NGP(scene.scale).cuda()
    g = torch.Generator().manual_seed(0)
    with torch.no_grad():
        p = m.xyz_encoder.params
        p[3072:] = ((torch.rand(p.numel() - 3072, generator=g) * 2 - 1) * 0.3).cuda()
        m.density_bitfield.copy_(torch.as_tensor(synth.pack_bits(synth.occupancy_grid(scene))).cuda())
    return m


def scene_by_name(which):
    return synth.lego_scene(0) if which == "lego" else synth.mip360_scene(0)


def render_target(n_rays):
    """the colour target of the render-parity losses"""
    return torch.rand(n_rays, 3, generator=torch.Generator().manual_seed(17)).cuda()


def composite_test_case():
    """inputs of one test-time compositing round: 150 of 200 rays alive, 8 samples each"""
    rng = np.random.RandomState(4)
    n_rays, n_alive, ns = 200, 150, 8
    alive = rng.permutation(n_rays)[:n_alive].astype(np.int64)
    sig = np.exp(rng.normal(0, 2.5, (n_alive, ns))).astype(np.float32)
    rgbs = rng.rand(n_alive, ns, 3).astype(np.float32)
    dl = np.full((n_alive, ns), 0.01, np.float32)
    ts = np.cumsum(dl, 1).astype(np.float32)
    neff = rng.randint(0, ns + 1, n_alive).astype(np.int32)
    op0 = (rng.rand(n_rays) * 0.9).astype(np.float32)
    dp0 = rng.rand(n_rays).astype(np.float32)
    rgb0 = rng.rand(n_rays, 3).astype(np.float32)
    return dict(alive=alive, sigmas=sig, rgbs=rgbs, deltas=dl, ts=ts, neff=neff, opacity=op0, depth=dp0, rgb=rgb0)


def loss_case(oracle):
    """NeRFLoss inputs: the oracle's compositing of a seeded ragged batch, and a seeded colour target"""
    c = composite_case(seed=12, n_rays=64, max_n=100)
    _, opacity, _, rgb, ws = oracle.composite_train_fw(c["sigmas"], c["rgbs"], c["deltas"], c["ts"], c["rays_a"], 1e-4)
    target = np.random.RandomState(13).rand(64, 3).astype(np.float32)
    return dict(rgb=rgb, opacity=opacity, ws=ws, deltas=c["deltas"], ts=c["ts"], rays_a=c["rays_a"], target=target)


def check_grads_vs_golden(model, g, prefix, tol):
    """the parameter gradients against a stored reference run (tests/golden/make_golden_parity.py): max |difference| below
    tol x the reference's largest magnitude, on rgb_net and the encoder MLP in full and on the stored hash-table entries"""
    p = dict(model.named_parameters())
    ga, gb = g[prefix + "g_rgb_net"], p["rgb_net.params"].grad.float().cpu().numpy()
    s = np.abs(ga).max()
    assert s > 0 and np.abs(ga - gb).max() < tol * s, "rgb_net.params grad: %g vs scale %g" % (np.abs(ga - gb).max(), s)
    gb = p["xyz_encoder.params"].grad.float().cpu().numpy()
    s = float(g[prefix + "g_xyz_scale"])
    idx = g[prefix + "g_xyz_idx"]
    err = max(np.abs(g[prefix + "g_xyz_mlp"] - gb[:3072]).max(), np.abs(g[prefix + "g_xyz_val"] - gb[idx]).max(),
              abs(np.abs(gb).max() - s))
    assert s > 0 and err < tol * s, "xyz_encoder.params grad: %g vs scale %g" % (err, s)


def check_view_vs_golden(res, g, prefix):
    """a test-time render against the stored rays of the reference's render of the same view"""
    idx = g[prefix + "idx"]
    for k in ("rgb", "opacity", "depth"):
        err = np.abs(res[k].detach().float().cpu().numpy()[idx] - g[prefix + k])
        assert err.max() < 2e-2 and err.mean() < 1e-3, "%s differs: max %g mean %g" % (k, err.max(), err.mean())
