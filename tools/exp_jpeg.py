"""Experiment: host (PIL) vs GPU (nvJPEG) texture decode time for the texture sizes of real scans."""
import io, sys, time, tempfile
from pathlib import Path
import numpy as np, torch
from PIL import Image
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from mvlm_b200 import build, synth
from mvlm_b200.io_obj import load_obj, _load_texture
build.build()
tmp = Path(tempfile.mkdtemp())
for size in (1024, 2048, 3072):
    tex = synth.face_texture(size, seed=1)
    Image.fromarray(tex).save(tmp / f"t{size}.jpg", quality=95)
    p = tmp / f"t{size}.obj"
    _load_texture(p, "nvjpeg", "cuda"); torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(5): a = np.asarray(Image.open(tmp / f"t{size}.jpg").convert("RGB"))
    t_pil = (time.perf_counter() - t0) / 5
    t0 = time.perf_counter()
    for _ in range(5): t, ev = _load_texture(p, "nvjpeg", "cuda")
    t_host = (time.perf_counter() - t0) / 5
    torch.cuda.synchronize(); t_all = (time.perf_counter() - t0) / 5
    d = np.abs(t.cpu().numpy().astype(int) - a.astype(int))
    print(f"{size}^2: PIL {t_pil*1e3:6.1f} ms | nvJPEG host part {t_host*1e3:6.1f} ms, incl. GPU {t_all*1e3:6.1f} ms | max diff {d.max()} mean {d.mean():.3f}")
