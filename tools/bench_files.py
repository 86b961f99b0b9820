"""From-files throughput with the host and the GPU OBJ parser (Pipeline(obj_parser=...)), beside the host-array e2e
figure of the same run.  Modelled on bench.py's e2e_files leg and run on the same seeded scan (grid 224: 50 176
vertices, 6.3 MB of OBJ text).

Per workload (views x image size, texture size):
  files[parser][decoder]  scans/s through Pipeline.predict_files (rank-local) or sharding.predict_files (torchrun),
                          variants alternated within the run, best of --rounds
  cpu_ms_per_scan         time.process_time of the whole process over the timed window, per scan
  e2e                     scans/s through Pipeline.predict_meshes(page-locked host arrays)
  gpu_parse_ms            CUDA events around the two phases of the device parser (file bytes already on the device;
                          includes the host round trip of the first phase's synchronisation)
Device name and power limit are read in the same call.

  python tools/bench_files.py [--out FILE]          one GPU
  torchrun --nproc-per-node 8 tools/bench_files.py  eight ranks (sharding.predict_files)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=32, help="scans per timed window (per rank)")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--workloads", default="100x256@1024,100x256@2048,8x256@1024")
    ap.add_argument("--out", type=Path)
    args = ap.parse_args()

    import torch.distributed as dist

    from mvlm_b200 import io_obj, sharding, synth
    from mvlm_b200.io_obj import Mesh
    from mvlm_b200.pipeline import create_pipeline
    from mvlm_b200.weights import seeded_state_dict

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank, local = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    def sync_max(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    verts, uvs, tris = synth.face_mesh(grid=224, seed=1234)
    sd = seeded_state_dict(N_LANDMARKS, "RGB+depth", 1234)
    results = []
    with tempfile.TemporaryDirectory() as tmp:
        for wl in args.workloads.split(","):
            shape, tex_size = wl.split("@")
            n_views, size = map(int, shape.split("x"))
            tex = synth.face_texture(int(tex_size), seed=1234)
            paths = [synth.write_obj(Path(tmp) / f"w{wl.replace('@', '_')}_{rank}_{i}.obj", verts, uvs, tris, tex)
                     for i in range(4)]
            dm = create_pipeline("dtu3d", n_views=n_views, weights=sd, seed=1234, verbose=False, image_size=(size, size),
                                 transforms=synth.random_view_transforms(n_views, seed=1234 + rank), device=f"cuda:{local}")
            hmesh = Mesh(*(torch.from_numpy(a).pin_memory().numpy() for a in (verts, tris, uvs, tex)))
            dm.predict_meshes([hmesh] * 4)
            n = args.files
            order = [(p, d) for p in ("host", "gpu") for d in ("pil", "nvjpeg")]
            best = {f"{p}/{d}": (0.0, None) for p, d in order}
            e2e = 0.0
            ref = None
            for rnd in range(args.rounds):
                if world > 1:
                    dist.barrier()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                dm.predict_meshes([hmesh] * n)
                torch.cuda.synchronize()
                e2e = max(e2e, world * n / sync_max(time.perf_counter() - t0))
                for p, d in (order if rnd % 2 == 0 else order[::-1]):
                    dm.obj_parser, dm.texture_decoder = p, d
                    dm.predict_files(paths[:2])  # warm-up of this variant (allocator pools, side streams, buffers)
                    batch = [str(paths[i % 4]) for i in range(n * world)]
                    if world > 1:
                        dist.barrier()
                    torch.cuda.synchronize()
                    c0, t0 = time.process_time(), time.perf_counter()
                    if world > 1:
                        out = sharding.predict_files(dm, batch)
                    else:
                        out = dict(enumerate(dm.predict_files(batch)))
                    torch.cuda.synchronize()
                    wall, cpu = time.perf_counter() - t0, time.process_time() - c0
                    rate = world * n / sync_max(wall)
                    if rate > best[f"{p}/{d}"][0]:
                        best[f"{p}/{d}"] = (rate, cpu * 1e3 / n)
                    lm = np.stack([out[k] for k in sorted(out)])
                    if p == "host" and d == "pil":
                        ref = lm
                    elif d == "pil":
                        assert np.array_equal(lm, ref), "landmarks differ between the parsers"
            # GPU parse time: bytes already on the device, events around the two phases on the loader stream
            st = io_obj.loader_state(dev)
            host = io_obj.read_pinned(paths[0], dev)
            text = host.to(dev)
            torch.cuda.synchronize()
            ms = []
            for _ in range(12):
                e0 = torch.cuda.Event(enable_timing=True)
                e0.record(st.stream)
                _, _, _, ready = io_obj.parse_obj_device(text, paths[0], dev)
                ready.synchronize()
                ms.append(e0.elapsed_time(ready))
            line = {
                "workload": {"views": n_views, "size": size, "texture": int(tex_size), "scan_obj_bytes": paths[0].stat().st_size},
                "ranks": world,
                "files_scans_per_s": {k: v[0] for k, v in best.items()},
                "cpu_ms_per_scan": {k: v[1] for k, v in best.items()},
                "e2e_scans_per_s": e2e,
                "gpu_parse_ms": {"median": float(np.median(ms[2:])), "min": float(np.min(ms[2:]))},
                "device": torch.cuda.get_device_name(dev),
                "power_limit_w": power_limit(local),
                "host_cores": os.cpu_count(),
                "files_per_window": n * world, "rounds": args.rounds,
            }
            results.append(line)
            if rank == 0:
                print(json.dumps(line), flush=True)
            del dm
            torch.cuda.empty_cache()
    if rank == 0 and args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        with open(args.out, "a") as f:
            for line in results:
                f.write(json.dumps(line) + "\n")
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
