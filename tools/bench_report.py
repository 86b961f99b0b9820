"""Cost of the per-landmark consensus report (DESIGN.md 7h) on one GPU.  Prints JSON lines (and appends them to --out):

  * the report kernel's device time: CUDA events around N consensus calls without and with the report, the
    difference per call, at C3 (73 landmarks x 100 views, H = 1) and C5 (84 x 200, H = 16 384);
  * predict_meshes scans/s at 8 and 100 views of 256^2, report off and on, alternated round by round.

The first line records the GPU's name and power limit, read in the same process."""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from mvlm_b200 import build, ops, synth  # noqa: E402
from mvlm_b200.io_obj import Mesh  # noqa: E402
from mvlm_b200.pipeline import create_pipeline  # noqa: E402
from mvlm_b200.weights import seeded_state_dict  # noqa: E402


def emit(out, **rec):
    line = json.dumps(rec)
    print(line, flush=True)
    if out is not None:
        with open(out, "a") as f:
            f.write(line + "\n")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def kernel_time(l, v, n_hyp, iters):
    peaks, starts, ends, _ = synth.synthetic_rays(l, v, outlier_frac=0.3, seed=1234)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    p, s, e = t(peaks), t(starts), t(ends)
    draws = t(synth.hypothesis_table(l, n_hyp, seed=1234).view(np.int32))
    ws = torch.empty((ops._lib.load().mvlm_consensus_workspace_bytes(l, v, n_hyp),), dtype=torch.uint8, device="cuda")
    res = {}
    for _ in range(2):  # alternate twice, keep the second round (warm)
        for report in (False, True):
            for _ in range(3):
                ops.consensus(p, s, e, draws, workspace=ws, report=report)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(iters):
                ops.consensus(p, s, e, draws, workspace=ws, report=report)
            b.record()
            b.synchronize()
            res[report] = a.elapsed_time(b) * 1e3 / iters
    return res[False], res[True]


def scans_per_second(dm, meshes, report, n):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    dm.predict_meshes(meshes[:n], report=report)
    torch.cuda.synchronize()
    return n / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", type=Path, default=None)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    build.build()
    emit(args.out, **gpu_info())
    for name, l, v, h, iters in (("C3", 73, 100, 1, 2000), ("C5", 84, 200, 16384, 200)):
        off, on = kernel_time(l, v, h, iters)
        emit(args.out, case=f"consensus {name} (L={l}, V={v}, H={h})", us_per_call_report_off=round(off, 2),
             us_per_call_report_on=round(on, 2), report_kernel_us=round(on - off, 2))
    vv, uv, tris = synth.face_mesh(grid=224, seed=1234)
    mesh = Mesh(verts=vv, tris=tris, uvs=uv, texture=synth.face_texture(1024, seed=1234))
    for n_views, n_scans in ((8, 64), (100, 16)):
        dm = create_pipeline("dtu3d", n_views=n_views, weights=seeded_state_dict(73, "RGB+depth", 1234), seed=1234,
                             verbose=False, image_size=(256, 256),
                             transforms=synth.random_view_transforms(n_views, seed=1234))
        meshes = [mesh] * n_scans
        for report in (False, True):  # warm-up: plans, graphs, pinned rings of both forms
            scans_per_second(dm, meshes, report, 4)
        rates = {False: [], True: []}
        for _ in range(args.rounds):
            for report in (False, True):
                rates[report].append(scans_per_second(dm, meshes, report, n_scans))
        emit(args.out, case=f"predict_meshes {n_views} views of 256^2, {n_scans} scans per round",
             scans_per_s_report_off=[round(x, 1) for x in rates[False]],
             scans_per_s_report_on=[round(x, 1) for x in rates[True]],
             median_off=round(float(np.median(rates[False])), 1), median_on=round(float(np.median(rates[True])), 1))


if __name__ == "__main__":
    main()
