"""Texture pages (texture_source="mtl", DESIGN.md 7g) on one GPU: load time, raster time and from-files throughput.

  load_ms[scan][parser][source]  ms per load_obj call, median of --repeats after one warm-up call: "single" = the
                                 bench face with one 1024^2 <stem>.jpg, "jpg" / "png" = the same face in 4 material
                                 groups with four 1024^2 JPEG / PNG pages; source "stem" = materials off, "mtl" = on
  raster_ms[scan][views]         CUDA events around render_device (256^2, mean of --repeats after a warm-up), the
                                 paged scans against the single texture
  files_scans_per_s[views]       Pipeline.predict_files over --scans copies, texture_source="mtl", host parser,
                                 variants alternated, best of --rounds
Device name and power limit are read in the same call.

  python tools/bench_mtl.py [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import shutil
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))


def device_info() -> dict:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, timeout=30)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": r.stdout.strip()}


def time_load(path: Path, parser: str, source: str, repeats: int) -> float:
    from mvlm_b200.io_obj import load_obj

    def once():
        t0 = time.perf_counter()
        m = load_obj(path, parser=parser, texture_source=source)
        for ev in (m.geometry_ready, m.texture_ready):
            if ev is not None:
                ev.synchronize()
        return time.perf_counter() - t0

    once()
    return 1e3 * statistics.median(once() for _ in range(repeats))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--scans", type=int, default=24)
    ap.add_argument("--out", type=Path)
    args = ap.parse_args()

    from mvlm_b200 import build, synth
    from mvlm_b200.io_obj import load_obj
    from mvlm_b200.pipeline import create_pipeline
    from mvlm_b200.weights import seeded_state_dict

    build.build()
    torch.cuda.set_device(0)
    lines = [{"info": device_info()}]
    tmp = Path(tempfile.mkdtemp(prefix="mvlm_mtl_bench_"))
    v, uv, t = synth.face_mesh(grid=224, seed=1234)
    groups = (np.arange(len(t)) * 4 // len(t)).astype(np.int32)
    pages = [synth.face_texture(1024, seed=1234 + i) for i in range(4)]
    scans = {"single": synth.write_obj(tmp / "single.obj", v, uv, t, pages[0]),
             "jpg": synth.write_obj_mtl(tmp / "jpg.obj", v, uv, t, pages, groups),
             "png": synth.write_obj_mtl(tmp / "png.obj", v, uv, t, pages, groups, formats=["png"] * 4)}
    row = {"load_ms": {k: {parser: {src: round(time_load(p, parser, src, args.repeats), 2) for src in ("stem", "mtl")}
                           for parser in ("host", "gpu")} for k, p in scans.items()}}
    lines.append(row)
    print(json.dumps(row), flush=True)

    kw = dict(weights=seeded_state_dict(73, "RGB+depth", 1234), seed=5, verbose=False, image_size=(256, 256))
    raster = {}
    for n_views in (8, 100):
        tr = synth.random_view_transforms(n_views, seed=3)
        dm = create_pipeline("dtu3d", n_views=n_views, transforms=tr, **kw)
        r = dm.renderer_3d
        for k in ("single", "jpg"):
            d = r.upload(load_obj(scans[k], texture_source="mtl"))
            r.render_device(d, tr)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(args.repeats * 3):
                r.render_device(d, tr)
            b.record()
            b.synchronize()
            raster.setdefault(k, {})[n_views] = round(a.elapsed_time(b) / (args.repeats * 3), 4)
    lines.append({"raster_ms": raster})
    print(json.dumps(lines[-1]), flush=True)

    for n_views in (8, 100):
        tr = synth.random_view_transforms(n_views, seed=3)
        dm = create_pipeline("dtu3d", n_views=n_views, transforms=tr, texture_source="mtl", **kw)
        paths = {k: [p] * args.scans for k, p in scans.items()}
        best = {k: 0.0 for k in paths}
        for rnd in range(args.rounds + 1):  # round 0 warms every plan, graph and buffer
            for k, ps in paths.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out = dm.predict_files(ps)
                torch.cuda.synchronize()
                rate = args.scans / (time.perf_counter() - t0)
                assert all(np.array_equal(o, out[0]) for o in out)
                if rnd > 0:
                    best[k] = max(best[k], rate)
        row = {"n_views": n_views, "image": 256, "scans": args.scans,
               "files_scans_per_s": {k: round(x, 1) for k, x in best.items()}}
        lines.append(row)
        print(json.dumps(row), flush=True)
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text("".join(json.dumps(x) + "\n" for x in lines))
    shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
