#!/usr/bin/env python
"""bench.py -- headline benchmark of the ngp_pl hot path on B200 (BASELINE.json metric: training rays/s,
plus 800x800 render FPS), one JSON line on rank 0.

    python bench.py --gpus 1 --steps K --warmup W            # this repo's sm_100a path
    python bench.py --impl reference ...                     # the reference's own path, same config
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   # N ranks, one per GPU
    python bench.py --workload c5 ...                        # BASELINE config 5 (unbounded, 6 cascades, 4096 rays)

Workloads (config.workload; both arms print the identical string):
  c2 (default): BASELINE config 2 -- Lego-shaped synthetic scene (no dataset on the box), 8192 rays/step per GPU,
      L=16 T=2^19 hash grid, 800x800 training images, Adam lr 1e-2 eps 1e-15, occupancy refresh every 16 steps.
  c5: BASELINE config 5 -- unbounded mip360-shaped synthetic scene, scale 16 (6 cascades), 4096 rays/step per GPU,
      exp_step_factor 1/256, black background.
Weak scaling (every rank draws its own batch, one gradient exchange per step). A "step" = batch assembly + march +
network forward + compositing + NeRFLoss + backward + gradient exchange + Adam, plus the occupancy refresh on its
cadence. The timed steps run after `--pretrain` untimed steps so the occupancy grid is in its steady state (the
reference's 30k-step headline is >99% steady-state steps); both arms do the same.

  value : whole-job rays/s with the image bank resident in HBM, CUDA-graph replay, CUDA events, max over ranks
  e2e   : the same step through Trainer.stage_batch()/train_step() with HOST (pinned) ray batches copied
          H2D every step and the loss scalars read back D2H (and waited for) every step
  render_fps : 800x800 test views sharded over the ranks (whole views, no communication), wall clock, max over ranks
  vren_ops   : the reference's twelve native operators one by one on a fixed seeded batch -- this repo's entries here,
               the reference's own compiled kernels in the `--impl reference` line (which also leaves its timings in
               gpurun_out/reference_arm_ops.json; when that file is present this line adds the per-operator ratios)
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_TRAIN_IMAGES = 100
REF_OPS_FILE = os.path.join(ROOT, "gpurun_out", "reference_arm_ops.json")

WORKLOADS = {
    "c2": dict(scene="lego", n_rays=8192,
               name="BASELINE config 2: Lego 800x800, 8192 rays/step/GPU, L=16 T=2^19 F=2, Adam lr 1e-2, "
                    "occupancy refresh every 16 steps"),
    "c5": dict(scene="mip360", n_rays=4096,
               name="BASELINE config 5: unbounded mip360-shaped synthetic scene 800x800, scale 16 (6 cascades), 4096 rays/step/GPU, "
                    "exp_step_factor 1/256, bg 0, L=16 T=2^19 F=2, Adam lr 1e-2, occupancy refresh every 16 steps"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--pretrain", type=int, default=None, help="untimed steps before the measurement")
    ap.add_argument("--fps-views", type=int, default=40, help="800x800 test views rendered for the FPS number (all ranks together)")
    ap.add_argument("--no-fps", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-vren-ops", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (per-ray rgb / opacity / depth / sample counts, the loss "
                         "terms, the fp32 parameters after its Adam update) to DIR/<name>.npy, for comparing two builds")
    ap.add_argument("--ref-tcnn", default="fast", choices=["fast", "standin"],
                    help="--impl reference: which tinycudann stand-in drives the reference's Python (fast = performance-grade)")
    ap.add_argument("--ddp", default="auto", choices=["auto", "p2p", "nvls", "p2p_host", "nccl", "zero"],
                    help="N>1 gradient exchange. p2p: ONE self-synchronising NVLink kernel (reduce-scatter + sharded Adam + "
                         "all-gather, in-kernel barriers, in the step's CUDA graph); nvls: the same through the NVSwitch multicast "
                         "mapping; p2p_host: round 1's host-barrier variant; zero: NCCL reduce_scatter/all_gather; nccl: "
                         "all-reduce + full Adam (the reference's DDP). auto = p2p up to 4 GPUs, nvls beyond")
    return ap.parse_args()


def make_scene(wl):
    from ngp_pl_b200 import synth
    return synth.lego_scene(0) if WORKLOADS[wl]["scene"] == "lego" else synth.mip360_scene(0)


# --------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """SM clock / throttle reasons DURING the timed region, sampled in-process through NVML every ~0.5 ms (the timed
    region of the driver's 20-step run is ~8 ms: nvidia-smi's 20 ms polling cannot land three samples in it).
    Falls back to `nvidia-smi -lms` rows when pynvml is missing."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []  # (time, sm_mhz, reasons bitmask)
        self.max_mhz = None
        self.t0 = self.t1 = None
        self._stop_evt = threading.Event()
        self.source = "nvml"

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            idx = self.index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                try:
                    idx = int(vis.split(",")[self.index])
                except (ValueError, IndexError):
                    idx = self.index
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            while not self._stop_evt.is_set():
                sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                except Exception:
                    rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                self.rows.append((time.time(), sm, rs))
                time.sleep(0.0005)
        except Exception:
            self.source = "nvidia-smi"
            self._run_smi()

    def _run_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                     "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in proc.stdout:
                if self._stop_evt.is_set():
                    proc.terminate()
                    break
                c = [x.strip() for x in line.split(",")]
                try:
                    mask = 0
                    for (nm, bit), v in zip(self.REASONS, c[2:6]):
                        if v.lower().startswith("active"):
                            mask |= bit
                    self.rows.append((time.time(), float(c[0]), mask))
                    self.max_mhz = float(c[1])
                except (ValueError, IndexError):
                    pass
        except Exception:
            pass

    def wait_first_row(self, timeout=5.0):
        t = time.time()
        while not self.rows and time.time() - t < timeout:
            time.sleep(0.01)

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        self._stop_evt.set()
        rows = [r for r in self.rows if self.t0 is not None and self.t0 <= r[0] <= (self.t1 or 1e30)]
        in_region = len(rows)
        if not rows:
            rows = self.rows[-3:]
        sm = [r[1] for r in rows]
        mask = 0
        for r in rows:
            mask |= r[2]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": [nm for nm, bit in self.REASONS if mask & bit], "samples": in_region, "source": self.source}


def dist_setup():
    import torch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    pg = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        pg = dist.group.WORLD
    return world, rank, local, pg


def barrier(world):
    import torch
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(x, world):
    import torch
    if world == 1:
        return x
    import torch.distributed as dist
    t = torch.tensor([x], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops", 1590.0)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


# --------------------------------------------------------------------------------------------------
def cpu_baseline_port(n_rays=16384):
    """The C oracle (a port: the reference has no CPU path) rendering a bounded sample of the same
    workload on one host core: march + network forward + compositing. Forward only -- the C oracle has no
    backward -- so this is an UPPER bound on what a CPU training step could reach."""
    import torch
    from oracle import oracle as O
    from ngp_pl_b200 import synth
    O.build()
    scene = synth.lego_scene(0)
    bits = synth.pack_bits(synth.occupancy_grid(scene))
    dirs = synth.ray_directions(synth.intrinsics())
    poses = torch.as_tensor(synth.camera_poses(N_TRAIN_IMAGES))
    rng = np.random.RandomState(0)
    img = torch.as_tensor(rng.randint(0, N_TRAIN_IMAGES, n_rays))
    pix = torch.as_tensor(rng.randint(0, dirs.shape[0], n_rays))
    o, d = synth.get_rays(dirs[pix], poses[img])
    o, d = o.numpy(), d.numpy()
    b = float(np.float32(np.exp(np.log(2048 * 0.5 / 16) / 15)))
    meta, entries = O.grid_meta(16, 19, 16, b)
    enc = rng.uniform(-0.1, 0.1, 3072 + 2 * entries).astype(np.float32)
    rgbp = rng.uniform(-0.2, 0.2, 7168).astype(np.float32)
    mn, mx = np.full((1, 3), -0.5, np.float32), np.full((1, 3), 0.5, np.float32)
    t0 = time.perf_counter()
    hits = O.ray_aabb(o, d, np.zeros(3, np.float32), np.full(3, 0.5, np.float32), 0.01)
    ra, xyzs, dd, deltas, ts = O.march_train(o, d, hits, bits, 1, 0.5, 0.0, rng.rand(n_rays).astype(np.float32), 128, 1024)
    sig, rgbs, _ = O.ngp_forward_c(meta, enc, rgbp, mn, mx, xyzs, dd)
    O.composite_train_fw(sig, rgbs, deltas, ts, ra, 1e-4)
    dt = time.perf_counter() - t0
    return {"value": n_rays / dt, "unit": "rays/s", "cores": 1, "kind": "port",
            "sample": "%d rays (%d samples) of the c2 workload, FORWARD render only (march + hash/MLP network + "
                      "compositing) by the C oracle on 1 host core, %.1f s; the reference has no CPU path and the oracle "
                      "has no backward, so this over-states CPU training throughput" % (n_rays, len(ts), dt)}


# --------------------------------------------------------------------------------------------------
# the reference's native operators, one by one, on a fixed seeded batch (both arms build the identical inputs)
# --------------------------------------------------------------------------------------------------
def time_vren_ops(vren, scene, dev):
    """vren: a module with the reference's twelve functions (reference models/csrc/binding.cpp:234-250) -- the reference's
    compiled extension, or ngp_pl_b200.vren. Median of 10 CUDA-event timings after 3 warm-up calls, per operator."""
    import torch
    from ngp_pl_b200 import synth
    n_rays, G = 8192, 128
    cascades, scale, esf = scene.cascades, float(scene.scale), float(scene.exp_step_factor)
    rng = np.random.RandomState(42)
    dirs = synth.ray_directions(synth.intrinsics())
    poses = torch.as_tensor(synth.camera_poses(N_TRAIN_IMAGES, radius=synth.camera_radius(scene), upper_only=scene.scale <= 0.5))
    img = torch.as_tensor(rng.randint(0, N_TRAIN_IMAGES, n_rays))
    pix = torch.as_tensor(rng.randint(0, dirs.shape[0], n_rays))
    o, d = synth.get_rays(dirs[pix], poses[img])
    o, d = o.to(dev).contiguous(), d.to(dev).contiguous()
    grid = torch.as_tensor(synth.occupancy_grid(scene)).to(dev)  # (cascades, G^3) in {0,1}
    bits = torch.as_tensor(synth.pack_bits(synth.occupancy_grid(scene))).to(dev)
    noise = torch.as_tensor(rng.rand(n_rays).astype(np.float32)).to(dev)
    center = torch.zeros(1, 3, device=dev)
    half = torch.full((1, 3), scale, device=dev)
    out = {}

    def timed(name, fn, setup=None, iters=10):
        ts_ = []
        for it in range(iters + 3):
            args = setup() if setup is not None else ()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); r = fn(*args); b.record()
            torch.cuda.synchronize()
            if it >= 3:
                ts_.append(a.elapsed_time(b))
        out[name] = float(np.median(ts_))
        return r

    _, hits_t, _ = timed("ray_aabb_intersect", lambda: vren.ray_aabb_intersect(o, d, center, half, 1))
    hits = hits_t[:, 0].contiguous()
    t0 = hits[:, 0]
    hits[:, 0] = torch.where((t0 >= 0) & (t0 < 0.01), torch.full_like(t0, 0.01), t0)
    rays_a, xyzs, dd, deltas, ts, counter = timed(
        "raymarching_train", lambda: vren.raymarching_train(o, d, hits, bits, cascades, scale, esf, noise, G, 1024))
    n = int(counter[0])
    deltas, ts = deltas[:n].contiguous(), ts[:n].contiguous()
    sig = torch.as_tensor(np.exp(rng.randn(n)).astype(np.float32) * 4).to(dev)
    rgbs = torch.as_tensor(rng.rand(n, 3).astype(np.float32)).to(dev)
    total, opacity, depth, rgb, ws = timed("composite_train_fw", lambda: vren.composite_train_fw(sig, rgbs, deltas, ts, rays_a, 1e-4))
    dLo = torch.as_tensor(rng.randn(n_rays).astype(np.float32)).to(dev)
    dLd = torch.zeros(n_rays, device=dev)
    dLc = torch.as_tensor(rng.randn(n_rays, 3).astype(np.float32)).to(dev)
    dLw = torch.zeros(n, device=dev)
    timed("composite_train_bw", lambda: vren.composite_train_bw(dLo, dLd, dLc, dLw, sig, rgbs, ws, deltas, ts, rays_a, opacity,
                                                               depth, rgb, 1e-4))
    _, wsi, wtsi = timed("distortion_loss_fw", lambda: vren.distortion_loss_fw(ws, deltas, ts, rays_a))
    dl = torch.ones(n_rays, device=dev)
    timed("distortion_loss_bw", lambda: vren.distortion_loss_bw(dl, wsi, wtsi, ws, deltas, ts, rays_a))
    bf = torch.zeros_like(bits)
    timed("packbits", lambda: vren.packbits(grid, 0.5, bf))
    coords = torch.as_tensor(rng.randint(0, G, (G ** 3 // 4, 3)).astype(np.int32)).to(dev)
    idx = timed("morton3D", lambda: vren.morton3D(coords))
    timed("morton3D_invert", lambda: vren.morton3D_invert(idx.int().contiguous()))
    # test-time operators on one full 800x800 view (640,000 rays), 4 samples per ray and round
    vo, vd = synth.get_rays(dirs, poses[0])
    vo, vd = vo.to(dev).contiguous(), vd.to(dev).contiguous()
    _, vh, _ = vren.ray_aabb_intersect(vo, vd, center, half, 1)
    vhits = vh[:, 0].contiguous()
    alive0 = torch.arange(vo.shape[0], device=dev)
    S = 4
    r = timed("raymarching_test", lambda h: vren.raymarching_test(vo, vd, h, alive0, bits, cascades, scale, esf, G, 1024, S),
              setup=lambda: (vhits.clone(),))
    _, _, tdel, tts, neff = r
    tsig = torch.as_tensor(np.exp(rng.randn(vo.shape[0], S)).astype(np.float32)).to(dev)
    trgb = torch.as_tensor(rng.rand(vo.shape[0], S, 3).astype(np.float32)).to(dev)
    timed("composite_test_fw",
          lambda h, al, op, dp, cl: vren.composite_test_fw(tsig, trgb, tdel, tts, h, al, 1e-4, neff, op, dp, cl),
          setup=lambda: (vhits.clone(), alive0.clone(), torch.zeros(vo.shape[0], device=dev), torch.zeros(vo.shape[0], device=dev),
                         torch.zeros(vo.shape[0], 3, device=dev)))
    return {"ms": out, "train_rays": n_rays, "train_samples": n, "test_rays": int(vo.shape[0]), "test_samples_per_ray": S}


def exchange_check(tr, world, rank):
    """First thing a multi-GPU run does: ONE optimiser step of the configured exchange against NCCL all_reduce + the
    full-size Adam kernel from identical state and per-rank random gradients (bitwise at N=2, 1e-6 beyond: only the fp32
    summation order differs); state is restored afterwards. Reported in the JSON line."""
    import torch
    import torch.distributed as dist
    from ngp_pl_b200 import _lib
    n = tr.n_params
    L = _lib.lib()
    st = torch.cuda.current_stream().cuda_stream
    state = [tr.P, tr.M, tr.V, tr.Ph, tr.step_dev] + list(tr._Gs)
    saved = [t.clone() for t in state]
    gcur = tr._gcur
    g = torch.Generator("cuda").manual_seed(4242 + rank)
    grad = torch.randn(n, device="cuda", generator=g) * 1e-3
    Pa, Ma, Va, Ga = tr.P.clone(), tr.M.clone(), tr.V.clone(), grad.clone()
    Pha = torch.empty(n, device="cuda", dtype=torch.float16)
    step_a = tr.step_dev.clone()
    dist.all_reduce(Ga)
    _lib.check(L.ngp_adam_step(Pa.data_ptr(), Ga.data_ptr(), Ma.data_ptr(), Va.data_ptr(), Pha.data_ptr(), n,
                               tr.lr_dev.data_ptr(), step_a.data_ptr(), tr.betas[0], tr.betas[1], tr.eps, 1.0 / world, 1, st), "adam")
    tr.G.copy_(grad)
    torch.cuda.synchronize()
    dist.barrier()
    tr.allreduce()
    tr.optimizer_step()
    torch.cuda.synchronize()
    lo, hi = tr.shard_bounds() if tr.ddp != "nccl" else (0, n)
    dP = (Pa[lo:hi] - tr.P[lo:hi]).abs().max().item()
    dH = (Pha.float() - tr.Ph.float()).abs().max().item()  # the WHOLE working copy: every peer's shard arrived
    t = torch.tensor([dP, dH], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dist.barrier()
    for a, b in zip(state, saved):
        a.copy_(b)
    tr._gcur = gcur
    torch.cuda.synchronize()
    dist.barrier()
    dP, dH = float(t[0]), float(t[1])
    # N = 2: bitwise (a + b == b + a). Beyond: only the fp32 summation order differs from NCCL's; a parameter that crosses an
    # fp16 rounding boundary moves the working copy by one fp16 ulp (<= 2^-10 of the parameter scale)
    scale = max(1.0, float(tr.P.abs().max()))
    tol, tol_half = (0.0, 0.0) if world == 2 else (2e-6 * scale, 2.0 ** -10 * scale)
    return {"against": "NCCL all_reduce + full-size ngp_adam_step", "max_abs_diff_params_owned_shard": dP,
            "max_abs_diff_fp16_working_copy": dH, "bitwise": dP == 0.0 and dH == 0.0, "ok": dP <= tol and dH <= tol_half,
            "tolerance": "bitwise" if world == 2 else "2e-6 on fp32 parameters, one fp16 ulp on the working copy (summation order)"}


# --------------------------------------------------------------------------------------------------
def make_trainer(args, scene, world, rank, pg, dev):
    """the workload's model, trainer and image bank in their seeded initial state"""
    from ngp_pl_b200 import synth
    from ngp_pl_b200.models.networks import NGP
    from ngp_pl_b200.trainer import Trainer
    bank = synth.RayBank(scene, n_images=N_TRAIN_IMAGES, device=dev, seed=rank)  # every rank: own images order/sampling
    # auto: the peer-load kernel up to 4 GPUs, the NVSwitch-reduced variant beyond (measured ms/step p2p vs nvls: N=2 0.390 vs
    # 0.425, N=4 0.381 vs 0.387, N=8 0.447 vs 0.431; profiles/r02_bench_n2_*.json, r02_exchange_residency.txt,
    # r02_bench_n8_*.json); falls back to p2p without a multicast mapping
    ddp_mode = args.ddp if args.ddp != "auto" else ("p2p" if world <= 4 else "nvls")
    tkw = dict(n_rays=WORKLOADS[args.workload]["n_rays"], lr=1e-2, exp_step_factor=scene.exp_step_factor, bg=(scene.bg,) * 3,
               process_group=pg, world_size=world, rank=rank, seed=rank)
    model = NGP(scene.scale).to(dev)
    try:
        tr = Trainer(model, ddp=ddp_mode, **tkw)
    except Exception as e:  # symmetric memory / multicast unavailable: fall back and say so in the line
        if world == 1 or ddp_mode not in ("p2p", "nvls", "p2p_host"):
            raise
        fallback = "p2p" if ddp_mode == "nvls" else "zero"
        ddp_note = "%s (%s unavailable: %s)" % (fallback, ddp_mode, type(e).__name__)
        model = NGP(scene.scale).to(dev)
        tr = Trainer(model, ddp=fallback, **tkw)
        ddp_mode = ddp_note
    tr.attach_bank(bank)
    return model, tr, bank, ddp_mode


def run_b200(args):
    import torch
    from ngp_pl_b200 import _lib
    from ngp_pl_b200.models.rendering import render
    world, rank, local, pg = dist_setup()
    dev = torch.device("cuda", local)
    wl = WORKLOADS[args.workload]
    n_rays = wl["n_rays"]
    scene = make_scene(args.workload)
    esf = scene.exp_step_factor
    model, tr, bank, ddp_mode = make_trainer(args, scene, world, rank, pg, dev)
    xchk = exchange_check(tr, world, rank) if world > 1 else None
    pretrain = args.pretrain if args.pretrain is not None else 1000
    K, W = args.steps, max(args.warmup, 3)
    sampler = ClockSampler(local)
    sampler.start()

    # CUDA graphs: [batch + march] / [network fwd + loss + bwd] / [Adam or the fused exchange]; the next step's [batch + march]
    # replays on a side stream while this step's compute + optimiser run
    tr.capture(sample=True)
    step = tr.train_step
    for _ in range(pretrain):
        step()
    for _ in range(W):
        step()
    barrier(world)
    sampler.wait_first_row()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(world)
    l0 = tr.launch_count()
    sampler.mark_begin()
    torch.cuda.profiler.start()  # `ncu --profile-from-start off ...` then sees exactly the timed steps (no-op otherwise)
    e0.record()
    for _ in range(K):
        step()
    e1.record()
    barrier(world)
    torch.cuda.profiler.stop()
    sampler.mark_end()
    launches = tr.launch_count() - l0
    ms = max_over_ranks(e0.elapsed_time(e1), world)
    clocks = sampler.stop()
    tr.check_exchange()
    stats = tr.stats()
    value = world * n_rays * K / (ms * 1e-3)

    # ---- e2e: host batches, H2D every step, loss read back (and waited for) every step ------------------
    n_host = 32
    host = [tuple(t.cpu().pin_memory() for t in bank.sample(n_rays)) for _ in range(n_host)]
    out_host = torch.zeros(8, dtype=torch.float32).pin_memory()
    tr.capture(sample=False)
    step_nosample = lambda: tr.train_step(sample=False)

    def e2e_step(i):
        # step i consumes the batch staged before; the NEXT batch's host->device copy and march are enqueued (side stream)
        # before this step's result is waited for, as any prefetching loader does -- every step still pays its own H2D
        # copy and its own loss read-back inside the timed region
        step_nosample()
        tr.stage_batch(*host[(i + 1) % n_host])
        out_host.copy_(tr.scalars, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return float(out_host[2])
    tr.stage_batch(*host[0])
    for i in range(W):
        e2e_step(i)
    barrier(world)
    e0.record()
    for i in range(K):
        e2e_step(i)
    e1.record()
    barrier(world)
    ms_e2e = max_over_ranks(e0.elapsed_time(e1), world)
    e2e = {"value": world * n_rays * K / (ms_e2e * 1e-3), "unit": "rays/s", "steps": K,
           "h2d_bytes_per_step": n_rays * 9 * 4, "d2h_bytes_per_step": 32}
    tr.check_exchange()

    # ---- roofline of the network kernels, timed alone with CUDA events (rank 0) -----------------------------
    roof = None
    if rank == 0:
        hbm, tf, which = peaks()
        n_samples = stats["rm_samples"]
        smp = _lib.NgpSamples()
        smp.rays_o, smp.rays_d = tr.rays_o.data_ptr(), tr.rays_d.data_ptr()
        smp.ray_idx, smp.ts = tr.ray_idx.data_ptr(), tr.ts.data_ptr()
        smp.n, smp.n_dev = tr.capacity, tr.counters[2:].data_ptr()
        # the backward visits only the composited samples (live list of the last step; counters[5] = its length)
        smp_b = _lib.NgpSamples.from_buffer_copy(smp)
        n_bwd = stats["bw_samples"]
        if tr.live_idx is not None:
            smp_b.live_idx, smp_b.n_live_dev = tr.live_idx.data_ptr(), tr.counters[5:].data_ptr()
        L = _lib.lib()
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

        def timed(fn, cold, iters=10):
            ts_ = []
            for it in range(iters + 3):
                if cold:
                    flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); fn(); b.record()
                torch.cuda.synchronize()
                if it >= 3:
                    ts_.append(a.elapsed_time(b))
            return float(np.mean(ts_))
        st = torch.cuda.current_stream().cuda_stream
        ws = (tr.bwd_ws.data_ptr(), tr.bwd_ws.numel())
        G = tr.G
        f_mlp = lambda: L.ngp_net_backward_mlp(C.byref(tr.net), C.byref(smp_b), tr.dsigmas.data_ptr(), tr.drgbs.data_ptr(),
                                               tr.feat_save.data_ptr(), tr.scalars[1:].data_ptr(), G.data_ptr(),
                                               G[tr.n_enc:].data_ptr(), ws[0], ws[1], st)
        f_sc = lambda: L.ngp_net_backward_scatter(C.byref(tr.net), C.byref(smp_b), tr.scalars[1:].data_ptr(), G.data_ptr(),
                                                  ws[0], ws[1], st)
        f_fwd = lambda: L.ngp_net_forward(C.byref(tr.net), C.byref(smp), 1, tr.sigmas.data_ptr(), tr.rgbs.data_ptr(),
                                          None, tr.feat_save.data_ptr(), st)
        # warm = back-to-back launches (table, gradient table and per-sample buffers in L2, as inside the step, where each
        # kernel runs right after its producer); cold = after a 256 MB L2 flush
        t = {k: {"warm": timed(f, False), "cold": timed(f, True)} for k, f in (("mlp", f_mlp), ("sc", f_sc), ("fwd", f_fwd))}
        G.zero_()
        traffic, traffic_src = {}, None
        prof = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(prof):
            try:
                traffic = json.load(open(prof))
                traffic_src = "profiles/ncu_traffic.json (%s): ncu --set full capture of a c2 step, NOT measured in this run" % \
                    traffic.get("_source", "capture")
            except Exception:
                traffic = {}

        def entry(kernel, bound, tt, n_, per_sample, peak, unit, note):
            alg = n_ * per_sample
            ms_ = tt["warm"]
            ach = alg / (ms_ * 1e-3) / (1e9 if unit == "GB/s" else 1e12)
            return {"kernel": kernel, "bound": bound, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
                    "traffic": traffic.get(kernel + "_dram_bytes_per_launch"), "ms_per_launch": ms_,
                    "ms_per_launch_cold_l2": tt["cold"], "samples_per_launch": n_, "algorithmic": note}
        # algorithmic work per sample (SURVEY.md section 8d / DESIGN.md): forward 512 B of table reads, scatter 1,024 B of
        # table-gradient read-modify-write, MLP backward 40,960 FLOP (dgrad + wgrad; the forward recompute is not counted)
        ks = [entry("k_ngp_fwd", "hbm", t["fwd"], n_samples, 512.0, hbm, "GB/s", "512 B/sample table gathers, every marched sample"),
              entry("k_grid_scatter_merged", "hbm", t["sc"], n_bwd, 1024.0, hbm, "GB/s",
                    "1,024 B/sample gradient RMW, composited samples only"),
              entry("k_ngp_bwd3", "tensor", t["mlp"], n_bwd, 40960.0, tf, "TFLOP/s",
                    "40,960 FLOP/sample dgrad (mma.sync) + wgrad (tcgen05.mma, TMEM accumulators), composited samples only")]
        roof = dict(max(ks, key=lambda e: e["ms_per_launch"]))  # the dominant kernel of the step
        roof["peak_source"] = which
        roof["traffic_source"] = traffic_src
        roof["kernels"] = ks
        roof["timing"] = "CUDA events around single launches on the current stream, mean of 10 after 3 warm-ups; ms_per_launch = warm L2 " \
                         "(in-step state), ms_per_launch_cold_l2 = after a 256 MB flush"
        roof["note"] = ("hash table (22.9 MB fp16) and its fp32 gradient (45.8 MB) are L2-resident on B200, so DRAM traffic stays far "
                        "below the algorithmic bytes; the physical limiters are L1 wavefronts of divergent 4-B gathers / 8-B reductions "
                        "and, for the MLP backward, the latency of its per-row dgrad chain (profiles/)")

    # ---- 800x800 render FPS with the trained model (BASELINE config 3), views sharded over the ranks ------------
    fps = None
    if not args.no_fps:
        try:
            fps = render_fps(lambda o, d: render(model, o, d, test_time=True, exp_step_factor=esf), scene, dev, args.fps_views,
                             world, rank)
        except Exception as e:  # a secondary number: never let it sink the bench line
            fps = {"unavailable": repr(e)}
    ops = None
    if rank == 0 and not args.no_vren_ops:
        try:
            from ngp_pl_b200 import vren
            ops = time_vren_ops(vren, scene, dev)
            ops["impl"] = "ngp_pl_b200.vren (libngp_b200.so)"
            if os.path.exists(REF_OPS_FILE):
                ref = json.load(open(REF_OPS_FILE))
                if ref.get("workload") == args.workload:
                    ops["reference_ms"] = ref["ms"]
                    ops["speedup_vs_reference_kernels"] = {k: ref["ms"][k] / v for k, v in ops["ms"].items() if k in ref["ms"] and v > 0}
                    ops["reference_source"] = "the reference's compiled models/csrc kernels (oracle/_ref), timed by `bench.py --impl " \
                                              "reference` on this box at %s" % ref.get("when", "?")
        except Exception as e:
            ops = {"unavailable": repr(e)}

    if args.dump_outputs:
        dump_outputs(args, scene, world, rank, pg, dev)
    if rank != 0:
        return
    line = {
        "metric": "train_rays_per_sec", "value": value, "unit": "rays/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16",
        "data": "synthetic (seeded %s-shaped box scene, 100 ray-traced 800x800 training views; random-init weights "
                "pre-trained %d untimed steps)" % (WORKLOADS[args.workload]["scene"], pretrain),
        "config": {"workload": wl["name"], "rays_per_step_per_gpu": n_rays, "global_rays_per_step": world * n_rays,
                   "parallelism": "dp%d" % world + ("" if world == 1 else " [%s]" % (
                       {"p2p": "one self-synchronising NVLink kernel: reduce-scatter + sharded Adam + all-gather, in the step's CUDA graph",
                        "nvls": "the same kernel through the NVSwitch multicast mapping (multimem.ld_reduce / multimem.st)",
                        "p2p_host": "NVLink reduce-scatter + Adam + all-gather kernel between host-launched barriers",
                        "zero": "NCCL reduce_scatter + sharded Adam + all_gather(fp16 params)",
                        "nccl": "NCCL all_reduce + full Adam"}.get(ddp_mode, ddp_mode))),
                   "pretrain_steps": pretrain,
                   "l2": "no explicit flush: each step streams params+grads+Adam moments (~230 MB) > 126 MB L2",
                   "samples_per_ray_marched": stats["rm_samples"] / n_rays, "samples_per_ray_composited": stats["vr_samples"] / n_rays,
                   "samples_per_ray_in_backward": stats["bw_samples"] / n_rays,
                   "train_psnr_last_batch": stats["psnr"]},
        "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
        "gpu_launches_how": "ngp_launch_count() delta over the timed region on rank 0: every launch recorded in a captured graph x its "
                            "replays + eager launches (occupancy refresh)",
        "roofline": roof,
    }
    if xchk is not None:
        line["exchange_check"] = xchk
    if fps is not None:
        line["render_fps"] = fps
    if ops is not None:
        line["vren_ops"] = ops
    if not args.no_cpu_baseline and world == 1:
        try:
            line["cpu_baseline"] = cpu_baseline_port()
        except Exception as e:  # the oracle is only a reported baseline; never let it sink the bench line
            line["cpu_baseline"] = {"unavailable": repr(e)}
    print(json.dumps(line))


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(args, scene, world, rank, pg, dev):
    """What one step of the timed path (Trainer.capture + train_step) hands its caller, as float32 .npy files in
    args.dump_outputs: per-ray rgb / opacity / depth / sample counts, the batch's target colours, the loss terms and the
    fp32 parameters after the Adam update. The step runs on a fresh trainer in the workload's seeded initial state, so its
    inputs are the same in every run and two builds can be compared output for output. (The trainer that was timed is not
    used: its gradient scatter accumulates with float atomics, and over the pretraining steps Adam amplifies those
    last-bit differences into a different trajectory in every run.) Rank 0 writes; every rank takes part in the step."""
    import torch
    _, tr, _, _ = make_trainer(args, scene, world, rank, pg, dev)
    tr.capture(sample=True)
    tr.train_step()
    if world > 1:
        tr.gather_master_params()
    torch.cuda.synchronize()
    if rank != 0:
        return
    out = {"rgb": tr.rgb, "opacity": tr.opacity, "depth": tr.depth, "n_samples": tr.n_samples, "loss_terms": tr.scalars,
           "rgb_gt": tr.rgb_gt, "params": tr.P}
    out = {k: v.detach().float().cpu().numpy() for k, v in out.items()}
    total = sum(a.nbytes for a in out.values())
    assert total <= DUMP_LIMIT_BYTES, "outputs of %d bytes exceed the %d-byte dump limit" % (total, DUMP_LIMIT_BYTES)
    os.makedirs(args.dump_outputs, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(args.dump_outputs, k + ".npy"), a)


def render_fps(render_fn, scene, dev, n_views, world=1, rank=0):
    """800x800 test views sharded over the ranks as whole views (no communication; the reference's validation loop renders
    one view per step per rank, train.py:193-237). FPS = views / wall time of the slowest rank, torch.cuda.synchronize()
    bracketed as in the reference's test.ipynb cell 2. One extra untimed view per rank warms up allocations."""
    import torch
    from ngp_pl_b200 import synth
    from ngp_pl_b200.trainer import shard_range
    K = synth.intrinsics()
    dirs = synth.ray_directions(K, dev)
    poses = torch.as_tensor(synth.camera_poses(n_views + 1, radius=synth.camera_radius(scene), seed=1234,
                                               upper_only=scene.scale <= 0.5)).to(dev)
    lo, hi = shard_range(n_views, world, rank)
    o, d = synth.get_rays(dirs, poses[n_views])
    res = render_fn(o, d)  # warm-up view
    samples = []
    barrier(world)
    t0 = time.perf_counter()
    for i in range(lo, hi):
        o, d = synth.get_rays(dirs, poses[i])
        res = render_fn(o, d)
        samples.append(res["total_samples"])
    torch.cuda.synchronize()
    dt = max_over_ranks(time.perf_counter() - t0, world)
    gt = synth.trace(scene, o, d)
    mse = ((res["rgb"].float() - gt) ** 2).mean().item()
    return {"value": n_views / dt, "unit": "frames/s", "resolution": "800x800", "views": n_views, "views_per_rank": hi - lo,
            "sharding": "whole views, contiguous ranges, no communication", "ms_per_frame_per_gpu": 1e3 * dt / max(hi - lo, 1),
            "samples_per_ray": float(sum(float(s) for s in samples) / max(len(samples), 1) / o.shape[0]),
            "psnr_last_view_rank0": -10 * float(np.log10(max(mse, 1e-12)))}


# --------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference's own path: its compiled vren kernels + its unmodified models/{rendering,networks,
    custom_functions}.py and losses.py (oracle/_ref), tinycudann replaced by a stand-in (tinycudann is unobtainable here:
    --ref-tcnn fast = performance-grade eager PyTorch, standin = the checker), driven by a loop that mirrors
    NeRFSystem.training_step (train.py:159-185) with fused torch.optim.Adam(eps=1e-15) in place of apex FusedAdam and a
    GradScaler like PL's precision=16. Same scene, config, pretrain and timing. A 1-GPU baseline: under torchrun only
    rank 0 runs."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref_env
    if not ref_env.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref (reference vren build) is not present on this box"}))
        return
    import torch
    torch.cuda.set_device(0)
    from ngp_pl_b200 import synth
    ref = ref_env.load_reference(tcnn=args.ref_tcnn)
    dev = torch.device("cuda", 0)
    wl = WORKLOADS[args.workload]
    n_rays = wl["n_rays"]
    scene = make_scene(args.workload)
    esf = scene.exp_step_factor
    rkw = {"exp_step_factor": esf} if esf else {}
    bank = synth.RayBank(scene, n_images=N_TRAIN_IMAGES, device=dev, seed=0)
    model = ref.NGP(scale=scene.scale).to(dev)
    G = model.grid_size
    model.register_buffer("density_grid", torch.zeros(model.cascades, G ** 3, device=dev))  # train.py:73-76
    gx = torch.stack(torch.meshgrid(*[torch.arange(G, dtype=torch.int32, device=dev)] * 3, indexing="ij"), -1).reshape(-1, 3)
    model.register_buffer("grid_coords", gx)
    opt = torch.optim.Adam(model.parameters(), lr=1e-2, eps=1e-15, fused=True)
    scaler = torch.amp.GradScaler("cuda")
    loss_fn = ref.losses.NeRFLoss(lambda_distortion=0)
    state = {"step": 0, "res": None}

    def step():
        # PL runs training_step under fp16 autocast with its GradScaler (Trainer(precision=16), train.py:274): the
        # network outputs are fp16, so without loss scaling the per-sample gradients underflow
        o, d, rgb = bank.sample(n_rays)  # fp32 rays (the reference builds them under autocast(dtype=float32), ray_utils.py:46)
        with torch.autocast("cuda", dtype=torch.float16):
            if state["step"] % 16 == 0:
                model.update_density_grid(0.01 * 1024 / 3 ** 0.5, warmup=state["step"] < 256)
            res = ref.render(model, o, d, **rkw)
            loss = sum(v.mean() for v in loss_fn(res, {"rgb": rgb}).values())
        opt.zero_grad(set_to_none=True)
        scaler.scale(loss).backward()
        scaler.step(opt)
        scaler.update()
        state["step"] += 1
        state["res"] = (res, rgb)
    pretrain = args.pretrain if args.pretrain is not None else 1000
    K, W = args.steps, max(args.warmup, 3)
    sampler = ClockSampler(0)
    sampler.start()
    for _ in range(pretrain + W):
        step()
    torch.cuda.synchronize()
    sampler.wait_first_row()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    sampler.mark_begin()
    e0.record()
    for _ in range(K):
        step()
    e1.record()
    torch.cuda.synchronize()
    sampler.mark_end()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    res, rgb = state["res"]
    mse = ((res["rgb"].float() - rgb) ** 2).mean().item()
    value = n_rays * K / (ms * 1e-3)
    tcnn_desc = {"fast": "performance-grade tinycudann STAND-IN (oracle/tcnn_fast.py: vectorised eager PyTorch, fp16 GEMMs, one gather / "
                         "one index_add_ per pass; tinycudann itself is unobtainable here, and its fused kernels are faster than this)",
                 "standin": "checker-grade tinycudann STAND-IN (oracle/tcnn_standin.py: per-level Python loop, fp32)"}[args.ref_tcnn]
    line = {
        "impl": "reference", "metric": "train_rays_per_sec", "value": value, "unit": "rays/s", "n_gpus": 1, "steps": K,
        "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16",
        "data": "synthetic (same scene/bank as the b200 arm), pre-trained %d untimed steps" % pretrain,
        "config": {"workload": wl["name"], "rays_per_step_per_gpu": n_rays, "global_rays_per_step": n_rays,
                   "parallelism": "dp1", "pretrain_steps": pretrain,
                   "stack": "reference vren CUDA kernels (compiled from /root/reference/models/csrc) + unmodified reference "
                            "render()/NGP/custom_functions/NeRFLoss + " + tcnn_desc + " + fused torch.optim.Adam (apex unavailable) + "
                            "GradScaler (PL precision=16)",
                   "samples_per_ray_marched": float(res["rm_samples"]) / n_rays,
                   "samples_per_ray_composited": float(res["vr_samples"]) / n_rays,
                   "train_psnr_last_batch": -10 * float(np.log10(max(mse, 1e-12)))},
        "clocks": clocks,
        "cpu_baseline": {"value": value, "unit": "rays/s", "cores": 0, "kind": "reference",
                         "sample": "the reference has NO CPU path (every op TORCH_CHECKs is_cuda); this is its own GPU path on the "
                                   "same B200, all %d steps of the workload" % K},
        "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if not args.no_fps:
        def ref_render(o, d):
            with torch.autocast("cuda", dtype=torch.float16):
                return ref.render(model, o, d, test_time=True, **rkw)
        line["render_fps"] = render_fps(ref_render, scene, dev, min(args.fps_views, 10))
    if not args.no_vren_ops:
        try:
            ops = time_vren_ops(ref.vren, scene, dev)
            ops["impl"] = "reference models/csrc kernels (oracle/_ref vren extension)"
            line["vren_ops"] = ops
            os.makedirs(os.path.dirname(REF_OPS_FILE), exist_ok=True)
            json.dump({"workload": args.workload, "ms": ops["ms"], "when": time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime())},
                      open(REF_OPS_FILE, "w"))
        except Exception as e:
            line["vren_ops"] = {"unavailable": repr(e)}
    print(json.dumps(line))


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
    try:
        import torch.distributed as _d
        if _d.is_initialized():
            _d.destroy_process_group()
    except Exception:
        pass
