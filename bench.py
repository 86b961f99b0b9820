#!/usr/bin/env python
"""Headline benchmark: scans/sec of the multi-view landmarking hot path (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # our arm (one rank per GPU via torchrun for N>1)
    python bench.py --impl reference --gpus N --steps K ...  # the CPU implementation of the same path

One "step" = one scan through the whole hot path: rasterise V views -> stacked-hourglass CNN ->
peaks -> rays -> RANSAC/LSQ consensus -> snap.  Workload = BASELINE.json configs[2] per GPU
(DTU3D RGB+depth, 100 views of 256^2, ~50k-vertex synthetic textured scan, seeded random-init
weights); scans shard over ranks with no data-path collective (weak scaling).

  value : scans/s with the scan already resident in HBM (CUDA events, max over ranks)
  e2e   : scans/s through the plugin call Pipeline.predict_meshes(host arrays) (batch form of predict_mesh):
          pinned-host -> device copies of every scan and the device -> host read of its (L,3) landmarks inside
          the timed region; sync_value = the same through one blocking predict_mesh call per scan
  roofline     : CNN stage (tensor-bound): algorithmic FLOPs (SURVEY.md 8d: 146.106 GFLOP/view) / event time
  cpu_baseline : the oracle port of the same path on the host cores, bounded sample, scaled to one scan (N = 1 only)
  --impl reference : the same port, every step one FULL scan on all host threads (nothing extrapolated)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

N_LANDMARKS = 73
IMAGE_MODE = "RGB+depth"
CPU_BUDGET_S = 45.0  # --impl reference: full scans are timed until this much CPU wall time is spent (at least one)


def config_dict(args, mesh, world):
    """The workload description; identical in both arms (the driver compares the dicts)."""
    return {"workload": f"DTU3D RGB+depth, {args.views} views {args.size}^2, {len(mesh.verts)} verts / {len(mesh.tris)} tris, "
                        "one scan per step per GPU",
            "n_landmarks": N_LANDMARKS, "ransac_hypotheses": args.hyp, "weights": "seeded random init",
            "l2": "per-step inputs + activations far exceed the 126 MB L2 (scan 5.4 MB, image stack 26 MB, CNN activations "
                  "of 100 views several GB); no explicit flush",
            "parallelism": f"scans sharded over {world} GPU(s), no collective"}


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm is meant to use the whole host."""
    import torch

    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        pass
    torch.set_num_threads(n)
    return torch.get_num_threads()


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--views", type=int, default=100)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--grid", type=int, default=224, help="mesh grid (224 -> 50 176 vertices / 99 458 triangles)")
    ap.add_argument("--hyp", type=int, default=1, help="RANSAC hypotheses per landmark (reference: 1)")
    ap.add_argument("--skip-cpu", action="store_true", help="omit the cpu_baseline leg")
    ap.add_argument("--profile", action="store_true", help="ncu mode: exact --warmup, no e2e / cpu legs")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path,
                    help="write the landmarks of the last timed step to DIR/landmarks.npy (float64; one file per rank "
                         "for N > 1) so that two builds can be compared on identical seeded inputs")
    ap.add_argument("--no-view-split", action="store_true", help="skip the config-4 leg (one scan's views split over the ranks)")
    ap.add_argument("--vs-views", type=int, default=200)
    ap.add_argument("--vs-size", type=int, default=512)
    ap.add_argument("--vs-grid", type=int, default=1001, help="1001 -> 1 002 001 vertices / 2 000 000 triangles")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def peaks_file():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return json.loads(p.read_text()), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """Streams nvidia-smi clocks / throttle reasons (100 ms period) during the timed region."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:  # noqa: BLE001
            self.proc = None

    def stop(self):
        samples = []
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
            except Exception:  # noqa: BLE001
                self.proc.kill()
                out = ""
            samples = [[x.strip() for x in ln.split(",")] for ln in out.splitlines() if ln.strip()]

        def num(x):
            try:
                return float(x)
            except ValueError:
                return None

        sm = [num(s[0]) for s in samples if num(s[0]) is not None]
        mx = [num(s[1]) for s in samples if len(s) > 1 and num(s[1]) is not None]
        pw = [num(s[2]) for s in samples if len(s) > 2 and num(s[2]) is not None]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s_ in samples:
            for k, n in enumerate(names):
                if len(s_) > 3 + k and s_[3 + k].lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(samples)}


def make_scan(args):
    from mvlm_b200 import synth
    from mvlm_b200.io_obj import Mesh

    verts, uvs, tris = synth.face_mesh(grid=args.grid, seed=1234)
    tex = synth.face_texture(1024, seed=1234)
    return Mesh(verts=verts, tris=tris, uvs=uvs, texture=tex)


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_path_seconds_per_scan(args, mesh, sample_views: int):
    """Times the oracle port (torch-CPU CNN restating the reference model, numpy peaks / rays /
    consensus restating the reference's numpy code, C restatements of the two VTK stages) on a
    bounded sample and scales it to one scan of `args.views` views."""
    import torch

    from mvlm_b200 import synth
    from mvlm_b200.weights import seeded_state_dict
    from oracle import native, stages
    from oracle.hourglass_ref import HourglassOracle

    v_all = args.views
    tr = synth.random_view_transforms(v_all, seed=1234)
    rot = stages.rotation_matrices(tr)
    t = {}
    t0 = time.perf_counter()
    img, _, _ = native.raster_multiview(mesh.verts, mesh.uvs, mesh.tris, mesh.texture, rot[:sample_views], args.size, args.size)
    t["raster"] = (time.perf_counter() - t0) / sample_views * v_all
    sd = seeded_state_dict(N_LANDMARKS, IMAGE_MODE, 1234)
    net = HourglassOracle(sd)
    x = torch.from_numpy(img).permute(0, 3, 1, 2).contiguous()
    t0 = time.perf_counter()
    hms = [net.forward(x[i:i + 2]) for i in range(0, sample_views, 2)]  # batch_size=2 as shipped
    t["cnn"] = (time.perf_counter() - t0) / sample_views * v_all
    hm = torch.cat(hms).numpy()
    t0 = time.perf_counter()
    pk = stages.heatmap_peaks(hm, "simple")
    t["peaks"] = (time.perf_counter() - t0) / sample_views * v_all
    # rays / consensus / snap at full size (cheap): tile the sampled peaks to all views
    reps = (v_all + sample_views - 1) // sample_views
    pk_all = np.tile(pk, (1, reps, 1))[:, :v_all]
    t0 = time.perf_counter()
    s, e = stages.landmark_lines(args.size, pk_all, tr)
    t["rays"] = time.perf_counter() - t0
    draws = synth.hypothesis_table(N_LANDMARKS, args.hyp, 1234)
    t0 = time.perf_counter()
    lm, _, _ = stages.landmarks_from_lines(pk_all, s, e, draws)
    t["consensus"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    native.snap_to_mesh(mesh.verts, mesh.tris, lm)
    t["snap"] = time.perf_counter() - t0
    return sum(t.values()), t, torch.get_num_threads()


def run_reference(args):
    """--impl reference: the CPU implementation of the path (oracle port; the reference tree and VTK
    are not present on the GPU box), all host threads, each step a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import native

    native.build()
    cores = use_all_host_threads()
    mesh = make_scan(args)
    n_warm = min(args.warmup, 1)
    for _ in range(n_warm):
        cpu_path_seconds_per_scan(args, mesh, 2)  # a short warm-up (thread pools, allocator), not a full scan
    # every timed step is ONE FULL scan (all views through raster / CNN / peaks, no extrapolation); full scans are
    # repeated until CPU_BUDGET_S is spent (about 15 s each on a 32-core host), at most --steps of them
    secs, parts = [], {}
    t_begin = time.perf_counter()
    while len(secs) < max(1, args.steps) and (not secs or time.perf_counter() - t_begin + secs[-1] < CPU_BUDGET_S):
        s, parts, _ = cpu_path_seconds_per_scan(args, mesh, args.views)
        secs.append(s)
    sec = float(np.mean(secs))
    val = 1.0 / sec
    line = {
        "impl": "reference", "metric": "scans/sec", "value": val, "unit": "scans/s", "n_gpus": args.gpus,
        "steps": len(secs), "warmup": n_warm, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args, mesh, args.gpus),
        "cpu_baseline": {"value": val, "unit": "scans/s", "cores": cores, "kind": "port",
                         "sample": f"{len(secs)} full scan(s) of {args.views} views, nothing extrapolated; the oracle port (torch-CPU "
                                   "restatement of MVLMModel, numpy peaks / rays / consensus restating the reference, C restatements "
                                   "of the two VTK stages: /root/reference and VTK do not exist on this box); stage seconds per scan: "
                                   + ", ".join(f"{k} {v:.2f}" for k, v in parts.items())},
        "e2e": {"value": val, "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ config 4
def run_view_split(args, world, rank, local, dev):
    """BASELINE.json config 4 under the driver: ONE scan (2M triangles, 200 views of 512^2) whose views are split over
    the ranks -- each rank rasterises and runs the CNN on its block, the fused arg-max writes the keys into the rank's
    slot of the gather buffer, one in-place NCCL all-gather, peaks / rays / consensus / snap on every rank
    (mvlm_b200/sharding.py::predict_mesh_view_split).  Strong scaling: the work per scan is fixed.  Reports ms/scan
    (CUDA events, max over ranks), the collective, the scan upload, the same scan on rank 0 alone in this run
    (N = 1 point of the curve) and whether a 32-view scan gives bit-identical landmarks both ways."""
    import torch
    import torch.distributed as dist

    from mvlm_b200 import ops, sharding, synth
    from mvlm_b200.io_obj import Mesh
    from mvlm_b200.pipeline import create_pipeline
    from mvlm_b200.weights import seeded_state_dict

    v_all, size = args.vs_views, args.vs_size
    verts, uvs, tris = synth.face_mesh(grid=args.vs_grid, seed=1234)
    mesh = Mesh(verts=verts, tris=tris, uvs=uvs, texture=synth.face_texture(1024, seed=1234))
    tr = synth.random_view_transforms(v_all, seed=77)
    sd = seeded_state_dict(N_LANDMARKS, IMAGE_MODE, 1234)
    dm = create_pipeline("dtu3d", n_views=v_all, weights=sd, seed=5, n_hypotheses=args.hyp, verbose=False,
                         image_size=(size, size), transforms=tr, device=f"cuda:{local}")

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, reps, warm):
        for _ in range(warm):
            out = fn()
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            out = fn()
        e1.record()
        sync_all()
        t = torch.tensor([e0.elapsed_time(e1) / reps], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), out

    res = {"workload": f"one scan, {len(verts)} verts / {len(tris)} tris, {v_all} views {size}^2, views split over {world} rank(s)",
           "scaling": "strong", "n_ranks": world}
    if world > 1:
        ms_split, lm_split = timed(lambda: sharding.predict_mesh_view_split(dm, mesh, tr), 5, 3)
        res["ms_per_scan"] = ms_split
        # the collective alone: in-place all-gather of the keys + the kernel that turns the gathered keys into peaks
        kb = dm.__dict__["_vs_keys"]
        ms_gather, _ = timed(lambda: (sharding.allgather_keys(kb), ops.peaks_from_gathered_keys(kb, v_all, size)), 20, 5)
        res["allgather_us"] = 1e3 * ms_gather
        res["allgather_bytes_per_rank"] = int(kb[0].numel() * 8)
        ms_up, _ = timed(lambda: sharding.upload_mesh_sharded(dm.renderer_3d, mesh), 5, 3)
        res["upload_ms"] = ms_up
        res["upload_bytes"] = int(sharding._mesh_bytes(mesh))
        # this rank's share of raster + CNN (what the split cannot remove)
        start, count = sharding.split_views(v_all, rank, world)
        dmesh = dm.renderer_3d.upload(mesh)

        def share():
            loc = dm.renderer_3d.render_device(dmesh, tr[start:start + count])
            dm.predictor_2d.predict_keys_device(loc["u8"], kb[rank, :count])

        ms_share, _ = timed(share, 5, 2)
        res["rank_raster_cnn_ms"] = ms_share
        res["overhead_ms"] = ms_split - ms_share
    # the same scan on one GPU (rank 0 alone; the other ranks wait): the N = 1 point of the strong-scaling curve
    sync_all()
    single_ms = None
    lm_single = None
    if rank == 0:
        for _ in range(2):
            lm_single = dm.predict_mesh(mesh)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            lm_single = dm.predict_mesh(mesh)
        e1.record()
        torch.cuda.synchronize()
        single_ms = e0.elapsed_time(e1) / 3
    sync_all()
    res["single_rank_ms"] = single_ms
    if world == 1:
        res["ms_per_scan"] = single_ms
    elif rank == 0:
        res["strong_scaling_efficiency"] = single_ms / (world * res["ms_per_scan"])
    # 32 views both ways: bit-identical landmarks
    if world > 1:
        tr32 = tr[:32]
        dm32 = create_pipeline("dtu3d", n_views=32, weights=sd, seed=5, n_hypotheses=args.hyp, verbose=False,
                               image_size=(size, size), transforms=tr32, device=f"cuda:{local}")
        a = sharding.predict_mesh_view_split(dm32, mesh, tr32)
        b = dm32.predict_mesh(mesh)
        flag = torch.tensor([int(np.array_equal(a, b))], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        res["equals_single_rank_32_views"] = bool(flag.item())
    del dm
    torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import torch
    import torch.distributed as dist

    from mvlm_b200 import _lib, build, synth
    from mvlm_b200.pipeline import create_pipeline
    from mvlm_b200.weights import seeded_state_dict

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    build.build()
    lib = _lib.load()
    dev = torch.device("cuda", local)

    mesh = make_scan(args)
    sd = seeded_state_dict(N_LANDMARKS, IMAGE_MODE, 1234)
    transforms = synth.random_view_transforms(args.views, seed=1234 + rank)
    dm = create_pipeline("dtu3d", n_views=args.views, weights=sd, seed=1234, n_hypotheses=args.hyp, verbose=False,
                         image_size=(args.size, args.size), transforms=transforms, device=f"cuda:{local}")
    r, p, e = dm.renderer_3d, dm.predictor_2d, dm.estimator_3d
    net = p.network(args.views, args.size, args.size)
    from mvlm_b200 import ops
    from mvlm_b200.utils.render3d import rotation_matrices

    dmesh = r.upload(mesh)
    rot = torch.from_numpy(rotation_matrices(transforms).reshape(-1, 9)).to(dev)
    draws = torch.from_numpy(e.seeded_draws(N_LANDMARKS).view(np.int32)).to(dev)
    zbuf = ops.raster_workspace(args.views, args.size, args.size, len(mesh.verts), dev)
    u8 = torch.empty((args.views, args.size, args.size, 4), dtype=torch.uint8, device=dev)
    ev = {k: (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for k in ("raster", "cnn", "tail")}

    def device_step(record=False):
        if record:
            ev["raster"][0].record()
        ops.raster_multiview(dmesh.verts, dmesh.uvs, dmesh.tris, dmesh.tex4(), rot, args.size, args.size, IMAGE_MODE,
                             zbuf=zbuf, out_u8=u8)
        if record:
            ev["raster"][1].record()
            ev["cnn"][0].record()
        peaks, _ = net.forward(u8, graph=True)
        if record:
            ev["cnn"][1].record()
            ev["tail"][0].record()
        starts, ends = ops.rays_from_peaks(peaks, rot, args.size)
        lm, err, _ = ops.consensus(peaks, starts, ends, draws)
        out, _ = ops.snap_to_mesh(dmesh.verts, dmesh.tris, lm)
        if record:
            ev["tail"][1].record()
        return out

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput
    n_warm = args.warmup if args.profile else max(args.warmup, 3)
    for _ in range(n_warm):
        device_step()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    lib.mvlm_launch_count(1)
    stage_ms = {k: 0.0 for k in ev}
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_start.record()
    pending = []
    for _ in range(args.steps):
        landmarks = device_step(record=True)
        # per-stage events are read after the loop; keep fresh pairs per step
        pending.append({k: ev[k] for k in ev})
        ev = {k: (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for k in ev}
    t_end.record()
    barrier()
    launches = lib.mvlm_launch_count(0)
    clocks = sampler.stop()
    ms_total = t_start.elapsed_time(t_end)
    for d in pending:
        for k, (a, b) in d.items():
            stage_ms[k] += a.elapsed_time(b)
    stage_ms = {k: v / args.steps for k, v in stage_ms.items()}
    tmax = torch.tensor([ms_total], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_total = float(tmax.item())
    value = world * args.steps / (ms_total / 1e3)
    if args.dump_outputs is not None:
        args.dump_outputs.mkdir(parents=True, exist_ok=True)
        name = "landmarks" if world == 1 else f"landmarks_rank{rank}"
        np.save(args.dump_outputs / f"{name}.npy", landmarks.cpu().numpy())

    # ---- end to end through the plugin call with host (pinned) buffers
    from mvlm_b200.io_obj import Mesh

    def pin(a):
        return None if a is None else torch.from_numpy(a).pin_memory().numpy()

    hmesh = Mesh(verts=pin(mesh.verts), tris=pin(mesh.tris), uvs=pin(mesh.uvs), texture=pin(mesh.texture))
    h2d = sum(a.nbytes for a in (hmesh.verts, hmesh.tris, hmesh.uvs, hmesh.texture)) + rot.numel() * 8 + draws.numel() * 4
    d2h = N_LANDMARKS * 3 * 8 + 8
    for _ in range(0 if args.profile else 2):
        dm.predict_mesh(hmesh)
    if not args.profile:
        dm.predict_meshes([hmesh] * 8)  # first use of the batch path grows the allocator pools (the copy stream has its own): warm-up, like the loop above
    barrier()
    n_e2e = 1 if args.profile else args.steps
    # (a) the batch form of the plugin call, Pipeline.predict_meshes: every scan's pinned-host -> device copies and its
    #     device -> host landmark read are inside the timed region; the next scan is enqueued while the previous runs
    t0 = time.perf_counter()
    res_all = dm.predict_meshes([hmesh] * n_e2e)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    res = res_all[-1]
    # (b) one synchronous predict_mesh call at a time (each call returns the landmarks before the next starts)
    barrier()
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        res_sync = dm.predict_mesh(hmesh)
    torch.cuda.synchronize()
    e2e_sync_s = time.perf_counter() - t0
    assert np.array_equal(res, res_sync)
    te = torch.tensor([e2e_s, e2e_sync_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * n_e2e / float(te[0].item())
    e2e_sync_value = world * n_e2e / float(te[1].item())
    assert res.shape == (N_LANDMARKS, 3) and np.isfinite(res).all()

    # ---- from files: Pipeline.predict_files(paths) = native multi-threaded OBJ parse + JPEG decode of the next scans
    #      on background threads while the GPU works (what predict_one_file(path) users get); informational
    files_value = files_nvjpeg_value = None
    if not args.profile:
        import tempfile

        with tempfile.TemporaryDirectory() as tmp:
            paths = []
            for i in range(4):
                paths.append(synth.write_obj(Path(tmp) / f"scan{rank}_{i}.obj", mesh.verts, mesh.uvs, mesh.tris, mesh.texture))
            n_files = max(8, min(args.steps, 32))
            dm.predict_files(paths[:2])
            barrier()
            t0 = time.perf_counter()
            out = dm.predict_files([paths[i % 4] for i in range(n_files)])
            torch.cuda.synchronize()
            tf = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(tf, op=dist.ReduceOp.MAX)
            files_value = world * n_files / float(tf.item())
            assert len(out) == n_files and all(o is not None and o.shape == (N_LANDMARKS, 3) for o in out)
            # same with the texture decoded on the GPU (nvJPEG, opt-in: pixel values differ slightly from libjpeg-turbo)
            dm.texture_decoder = "nvjpeg"
            dm.predict_files(paths[:2])
            barrier()
            t0 = time.perf_counter()
            out = dm.predict_files([paths[i % 4] for i in range(n_files)])
            torch.cuda.synchronize()
            tf = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(tf, op=dist.ReduceOp.MAX)
            files_nvjpeg_value = world * n_files / float(tf.item())
            dm.texture_decoder = "pil"

    view_split = None
    if not args.profile and not args.no_view_split:
        try:
            view_split = run_view_split(args, world, rank, local, dev)
        except Exception as ex:  # noqa: BLE001  (the headline numbers above stand on their own)
            view_split = {"error": f"{type(ex).__name__}: {ex}"}
    if rank == 0:
        pk, pk_kind = peaks_file()
        flops_scan = net.flops_per_view * args.views
        ach = flops_scan / (stage_ms["cnn"] / 1e3) / 1e12
        peak = pk["bf16_tflops_sustained"]
        line = {
            "metric": "scans/sec", "value": value, "unit": "scans/s", "n_gpus": world, "steps": args.steps,
            "warmup": n_warm, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": config_dict(args, mesh, world),
            "cnn_workspace_gb": lib.mvlm_hourglass_workspace_bytes(N_LANDMARKS, 4, args.views, args.size, args.size) / 1e9,
            "e2e": {"value": e2e_value, "unit": "scans/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "api": "Pipeline.predict_meshes(host meshes): up to two scans in flight on one stream",
                    "sync_value": e2e_sync_value,
                    "sync_api": "Pipeline.predict_mesh(host mesh), one blocking call per scan"},
            "e2e_files": {"value": files_value, "nvjpeg_value": files_nvjpeg_value, "unit": "scans/s",
                          "note": "Pipeline.predict_files(paths): .obj (6.3 MB text) + .jpg read from disk per scan, native "
                                  "multi-threaded parser, 2-deep prefetch; informational, not the contract's e2e"},
            "gpu_launches": int(launches),
            "stages_ms": stage_ms,
            "roofline": {"bound": "tensor", "kernel": "conv_flow_kernel + conv_umma_kernel (CNN stage: all its launches)",
                         "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": None,
                         "peak_source": f"{pk_kind} bf16_tflops_sustained", "flops_per_scan": flops_scan},
            "clocks": clocks,
            "view_split": view_split,
        }
        if world == 1 and not args.skip_cpu and not args.profile:
            try:
                cores = use_all_host_threads()
                n_sample = 8
                sec, parts, _ = cpu_path_seconds_per_scan(args, mesh, n_sample)
                line["cpu_baseline"] = {
                    "value": 1.0 / sec, "unit": "scans/s", "cores": cores, "kind": "port",
                    "sample": "%d of %d views for raster/CNN/peaks (scaled linearly), full size for rays/consensus/snap; "
                              "VTK stages restated in C, not executed; stage s/scan: %s" % (
                                  n_sample, args.views, ", ".join(f"{k} {v:.2f}" for k, v in parts.items()))}
            except Exception as ex:  # noqa: BLE001
                line["cpu_baseline"] = {"value": None, "unit": "scans/s", "cores": 0, "kind": "port", "sample": f"failed: {ex}"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
