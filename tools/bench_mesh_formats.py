"""PLY / STL scan loading and from-files throughput (one GPU).

  load[format][parser]  ms per load_ply_stl call: "host" = csrc/mesh_loader.cu, "gpu" = csrc/mesh_parse.cu (read into
                        page-locked memory, decode + weld on the device, host clock stopped after the result's event
                        has completed); median of --repeats, after one warm-up call per variant
  files[input]          scans/s through Pipeline.predict_files over --scans copies of one scan: binary STL (host and
                        GPU decoder), the same triangles as an untextured OBJ (host and GPU parser), and
                        Pipeline.predict_meshes over page-locked host arrays ("arrays"); variants alternated, best of
                        --rounds
Workloads: the bench face (grid 224: 50 176 vertices, 99 458 triangles) and the config-4 grid (1001: 2M triangles) for
the loads; 8 and 100 views of 256^2 for the throughput.  Device name and power limit are read in the same call.

  python tools/bench_mesh_formats.py [--out FILE]
"""
from __future__ import annotations

import argparse
import json
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


def time_load(path: Path, parser: str, repeats: int) -> float:
    from mvlm_b200.io_mesh import load_ply_stl

    def once():
        t0 = time.perf_counter()
        m = load_ply_stl(path, parser=parser)
        if m.geometry_ready is not None:
            m.geometry_ready.synchronize()
        return time.perf_counter() - t0, m

    _, m = once()
    if parser == "gpu":
        assert isinstance(m.verts, torch.Tensor), f"{path} took the host fallback"
    return 1e3 * statistics.median(once()[0] for _ in range(repeats))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--scans", type=int, default=24)
    ap.add_argument("--out", type=Path)
    args = ap.parse_args()

    from mvlm_b200 import build, synth
    from mvlm_b200.io_obj import Mesh, load_obj
    from mvlm_b200.pipeline import create_pipeline
    from mvlm_b200.weights import seeded_state_dict

    build.build()
    torch.cuda.set_device(0)
    lines = [{"info": device_info()}]
    tmp = Path(tempfile.mkdtemp(prefix="mvlm_mesh_bench_"))
    for grid in (224, 1001):
        v, _, t = synth.face_mesh(grid=grid, seed=1234)
        files = {"stl": synth.write_stl(tmp / f"g{grid}.stl", v, t),
                 "ply": synth.write_ply(tmp / f"g{grid}.ply", v, t)}
        row = {"grid": grid, "n_tris": int(len(t)), "load_ms": {}}
        for fmt, p in files.items():
            row["load_ms"][fmt] = {parser: round(time_load(p, parser, args.repeats), 3) for parser in ("host", "gpu")}
            row["load_ms"][fmt]["mbytes"] = round(p.stat().st_size / 1e6, 2)
        lines.append(row)
        print(json.dumps(row), flush=True)

    v, _, t = synth.face_mesh(grid=224, seed=1234)
    plain = load_obj(synth.write_obj(tmp / "plain.obj", v, None, t))  # the coordinates an OBJ file holds
    stl_paths = [synth.write_stl(tmp / f"s{i:03d}.stl", plain.verts, plain.tris) for i in range(args.scans)]
    obj_paths = [synth.write_obj(tmp / f"o{i:03d}.obj", plain.verts, None, plain.tris) for i in range(args.scans)]
    arrays = Mesh(verts=torch.from_numpy(plain.verts).pin_memory().numpy(),
                  tris=torch.from_numpy(plain.tris).pin_memory().numpy(), uvs=None, texture=None)
    for n_views in (8, 100):
        kw = dict(n_views=n_views, weights=seeded_state_dict(73, "RGB+depth", 1234), seed=5, verbose=False,
                  image_size=(256, 256), transforms=synth.random_view_transforms(n_views, seed=3))
        pipes = {"stl_host": (create_pipeline("dtu3d", scan_formats=("stl",), **kw), stl_paths),
                 "stl_gpu": (create_pipeline("dtu3d", scan_formats=("stl",), obj_parser="gpu", **kw), stl_paths),
                 "obj_host": (create_pipeline("dtu3d", **kw), obj_paths),
                 "obj_gpu": (create_pipeline("dtu3d", obj_parser="gpu", **kw), obj_paths),
                 "arrays": (create_pipeline("dtu3d", **kw), None)}
        ref = None
        best = {k: 0.0 for k in pipes}
        for rnd in range(args.rounds + 1):  # round 0 warms every plan, graph and buffer
            for name, (dm, paths) in pipes.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out = dm.predict_files(paths) if paths else dm.predict_meshes([arrays] * args.scans)
                torch.cuda.synchronize()
                rate = args.scans / (time.perf_counter() - t0)
                if ref is None:
                    ref = out[0]
                assert np.array_equal(out[-1], ref), f"{name}: landmarks differ from stl_host"
                if rnd > 0:
                    best[name] = max(best[name], rate)
        row = {"n_views": n_views, "image": 256, "scans": args.scans, "files_scans_per_s": {k: round(x, 1) for k, x in best.items()}}
        lines.append(row)
        print(json.dumps(row), flush=True)
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
