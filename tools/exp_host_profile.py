"""Experiment: host-side cost of one blocking predict_mesh call (cProfile, headline workload)."""
import cProfile, pstats, sys, time
from pathlib import Path
import numpy as np, torch
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from mvlm_b200 import build, synth
from mvlm_b200.io_obj import Mesh
from mvlm_b200.pipeline import create_pipeline
from mvlm_b200.weights import seeded_state_dict
build.build()
v, uv, t = synth.face_mesh(grid=224, seed=1234)
tex = synth.face_texture(1024, seed=1234)
pin = lambda a: torch.from_numpy(a).pin_memory().numpy()
mesh = Mesh(verts=pin(v), tris=pin(t), uvs=pin(uv), texture=pin(tex))
tr = synth.random_view_transforms(100, seed=1234)
dm = create_pipeline("dtu3d", n_views=100, weights=seeded_state_dict(73, "RGB+depth", 1234), seed=1234, verbose=False, image_size=(256, 256), transforms=tr)
for _ in range(3): dm.predict_mesh(mesh)
torch.cuda.synchronize()
t0 = time.perf_counter()
for _ in range(20): dm.predict_mesh(mesh)
print(f"blocking calls: {20/(time.perf_counter()-t0):.1f} scans/s")
t0 = time.perf_counter()
hs = [dm._enqueue_pass([mesh]) for _ in range(20)]
t_enq = time.perf_counter() - t0
torch.cuda.synchronize()
print(f"enqueue only: {t_enq/20*1e3:.2f} ms per scan of host time; all done after {(time.perf_counter()-t0)/20*1e3:.2f} ms per scan")
pr = cProfile.Profile(); pr.enable()
for _ in range(20): dm.predict_mesh(mesh)
pr.disable()
st = pstats.Stats(pr); st.sort_stats("cumulative").print_stats(22)
