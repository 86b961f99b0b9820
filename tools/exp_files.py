"""Experiment: where does the host time of the batch drivers go?  (GPU box)"""
import sys, time, tempfile
from pathlib import Path
import numpy as np, torch
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from mvlm_b200 import build, synth
from mvlm_b200.io_obj import Mesh, load_obj
from mvlm_b200.pipeline import create_pipeline
from mvlm_b200.weights import seeded_state_dict
build.build()
v, uv, t = synth.face_mesh(grid=224, seed=1234)
tex = synth.face_texture(1024, seed=1234)
tmp = Path(tempfile.mkdtemp())
paths = [synth.write_obj(tmp / f"s{i}.obj", v, uv, t, tex) for i in range(4)]
tr = synth.random_view_transforms(100, seed=1234)
dm = create_pipeline("dtu3d", n_views=100, weights=seeded_state_dict(73, "RGB+depth", 1234), seed=1234, verbose=False, image_size=(256, 256), transforms=tr)
meshes = [load_obj(p) for p in paths]
pinned = Mesh(*[torch.from_numpy(np.array(a)).pin_memory().numpy() for a in (meshes[0].verts, meshes[0].tris, meshes[0].uvs, meshes[0].texture)])
dm.predict_meshes([meshes[0], pinned])
enq, fin = [], []
oe, of = dm._enqueue_pass, dm._finish_pass
def e2(m, tr=None, **kw):
    t0 = time.perf_counter(); r = oe(m, tr, **kw); enq.append(time.perf_counter() - t0); return r
def f2(h, d, k):
    t0 = time.perf_counter(); r = of(h, d, k); fin.append(time.perf_counter() - t0); return r
dm._enqueue_pass, dm._finish_pass = e2, f2
for name, batch in (("same pinned mesh", [pinned] * 16), ("same pageable mesh", [meshes[0]] * 16), ("4 pageable meshes", [meshes[i % 4] for i in range(16)])):
    for depth in (1, 2):
        enq.clear(); fin.clear()
        torch.cuda.synchronize(); t0 = time.perf_counter()
        dm.predict_meshes(batch, depth=depth)
        torch.cuda.synchronize(); dt = time.perf_counter() - t0
        print(f"{name:20s} depth {depth}: {16/dt:5.1f} scans/s; enqueue {np.mean(enq)*1e3:5.2f} ms (max {np.max(enq)*1e3:5.2f}), finish wait {np.mean(fin)*1e3:5.2f} ms")
dm._enqueue_pass, dm._finish_pass = oe, of
import mvlm_b200.pipeline.general_pipeline as gp
orig = gp.load_obj
for nt in (0, 4):
    gp.load_obj = lambda f, nt=nt: orig(f, n_threads=nt)
    for pf in (1, 2, 3, 4):
        dm.predict_files(paths[:2], prefetch=pf)
        torch.cuda.synchronize(); t0 = time.perf_counter()
        dm.predict_files([paths[i % 4] for i in range(24)], prefetch=pf)
        torch.cuda.synchronize(); print(f"predict_files parser threads={nt or 16} prefetch={pf}: {24/(time.perf_counter()-t0):.1f} scans/s")
