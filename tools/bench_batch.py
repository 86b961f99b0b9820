"""Several scans in one device pass: is the CNN cheaper per scan when an 8-view plan carries 8*S views?

  --cnn   ops.Hourglass (73 landmarks, RGB+depth, 256^2) for n_views = 8*S, S in --scans; CUDA-graph replay timed with
          CUDA events after a warm-up, best and mean of --windows windows; reports ms per pass and per scan.
  --e2e   scans/s of the batch drivers on the bench scan (grid 224, 1024^2 texture) with one scan per pass (batching
          off: PASS_PIXELS = 0) and with the planner's pass size for --pass-pixels, the two arms alternated within the run, best of
          --rounds windows of --files scans each: device-resident meshes and page-locked host arrays through
          predict_meshes, OBJ files through predict_files with the host and the GPU parser (nvJPEG textures).  The
          landmarks of the two arms are checked to be bit-identical.  Workloads: 8 views (the preset) and 100 views
          (given random views) of 256^2.

Device name and power limit are read in the same call.  One JSON line per configuration goes to stdout and, with --out,
is appended to that file.

  python tools/bench_batch.py --cnn [--out profiles/batch_8views_1gpu.jsonl]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

N_LANDMARKS = 73


def power_limit(index: int):
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", str(index)],
                           capture_output=True, text=True, timeout=30)
        return float(r.stdout.strip())
    except Exception:  # noqa: BLE001
        return None


def device_info():
    return {"device": torch.cuda.get_device_name(0), "power_limit_w": power_limit(0)}


def cnn_leg(scans, views: int, size: int, iters: int, windows: int):
    from mvlm_b200 import ops

    sd = seeded_state_dict_cached()
    out = []
    for s in scans:
        v = views * s
        net = ops.Hourglass(sd, N_LANDMARKS, 4, v, size, size)
        img = torch.randint(0, 256, (v, size, size, 4), dtype=torch.uint8, device="cuda")
        for _ in range(5):
            net.forward(img, graph=True)
        torch.cuda.synchronize()
        ts = []
        for _ in range(windows):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                net.forward(img, graph=True)
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) / iters)
        line = {"leg": "cnn", "scans_per_pass": s, "views_per_scan": views, "size": size, "n_views": v,
                "ms_per_pass_best": min(ts), "ms_per_pass_mean": sum(ts) / len(ts),
                "ms_per_scan_best": min(ts) / s, "ms_per_scan_mean": sum(ts) / len(ts) / s,
                "iters_per_window": iters, "windows": windows, **device_info()}
        print(json.dumps(line), flush=True)
        out.append(line)
        del net, img
        torch.cuda.empty_cache()
    return out


def e2e_leg(views: int, size: int, n_files: int, rounds: int, pass_pixels: int):
    import tempfile

    import numpy as np

    from mvlm_b200 import synth
    from mvlm_b200.io_obj import Mesh
    from mvlm_b200.pipeline import create_pipeline
    from mvlm_b200.pipeline import general_pipeline as gp

    planned_pixels = gp.PASS_PIXELS
    verts, uvs, tris = synth.face_mesh(grid=224, seed=1234)
    tex = synth.face_texture(1024, seed=1234)
    sd = seeded_state_dict_cached()
    tr = None if views == 8 else synth.random_view_transforms(views, seed=1234)
    dm = create_pipeline("dtu3d", n_views=views, weights=sd, seed=1234, verbose=False, image_size=(size, size),
                         transforms=tr, texture_decoder="nvjpeg")
    pinned = Mesh(*(torch.from_numpy(a).pin_memory().numpy() for a in (verts, tris, uvs, tex)))
    device = Mesh(*(torch.from_numpy(a).cuda() for a in (verts, tris, uvs, tex)))
    with tempfile.TemporaryDirectory() as tmp:
        paths = [str(synth.write_obj(Path(tmp) / f"s{i}.obj", verts, uvs, tris, tex)) for i in range(4)]
        sources = {
            "device": lambda: dm.predict_meshes([device] * n_files),
            "pinned_host": lambda: dm.predict_meshes([pinned] * n_files),
            "files_host_parser": lambda: dm.predict_files([paths[i % 4] for i in range(n_files)]),
            "files_gpu_parser": lambda: dm.predict_files([paths[i % 4] for i in range(n_files)]),
        }
        arms = {"one_scan_per_pass": 0, "planner": pass_pixels}
        best = {(src, arm): 0.0 for src in sources for arm in arms}
        landmarks = {}
        for rnd in range(rounds):
            for src, run in sources.items():
                dm.obj_parser = "gpu" if src == "files_gpu_parser" else "host"
                for arm, pixels in (list(arms.items()) if rnd % 2 == 0 else list(arms.items())[::-1]):
                    gp.PASS_PIXELS = pixels
                    if rnd == 0:
                        run()  # warm-up: plans, graphs, pinned rings of this pass size
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    res = run()
                    torch.cuda.synchronize()
                    best[(src, arm)] = max(best[(src, arm)], n_files / (time.perf_counter() - t0))
                    lm = np.stack(res)
                    ref = landmarks.setdefault(src, lm)
                    assert np.array_equal(lm, ref), f"landmarks differ between the arms ({src})"
        gp.PASS_PIXELS = pass_pixels
        line = {"leg": "e2e", "views": views, "size": size, "pass_pixels": pass_pixels,
                "scans_per_pass": dm._scans_per_pass(),
                "scans_per_s": {f"{src}/{arm}": round(best[(src, arm)], 2) for src in sources for arm in arms},
                "speedup": {src: round(best[(src, "planner")] / best[(src, "one_scan_per_pass")], 3) for src in sources},
                "landmarks_bit_identical_between_arms": True, "texture_decoder": "nvjpeg",
                "files_per_window": n_files, "rounds": rounds, "host_cores": os.cpu_count(), **device_info()}
        gp.PASS_PIXELS = planned_pixels
    print(json.dumps(line), flush=True)
    del dm
    torch.cuda.empty_cache()
    return [line]


_SD = None


def seeded_state_dict_cached():
    global _SD
    if _SD is None:
        from mvlm_b200.weights import seeded_state_dict

        _SD = seeded_state_dict(N_LANDMARKS, "RGB+depth", 1234)
    return _SD


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cnn", action="store_true", help="CNN time per scan against scans per pass")
    ap.add_argument("--e2e", action="store_true", help="batch-driver throughput, batching off against the planner")
    ap.add_argument("--files", type=int, default=96, help="scans per timed window of --e2e at 8 views (24 at 100)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--pass-pixels", type=int, default=96 * 256 * 256, help="pixel budget of a pass in the planner arm")
    ap.add_argument("--scans", default="1,2,4,8,12,16")
    ap.add_argument("--views", type=int, default=8)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--iters", type=int, default=40)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--out", type=Path)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    lines = []
    if args.cnn:
        lines += cnn_leg([int(x) for x in args.scans.split(",")], args.views, args.size, args.iters, args.windows)
    if args.e2e:
        lines += e2e_leg(8, 256, args.files, args.rounds, args.pass_pixels)
        lines += e2e_leg(100, 256, max(8, args.files // 4), args.rounds, args.pass_pixels)
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
