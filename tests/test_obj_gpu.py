"""GPU: the opt-in device OBJ parser (csrc/obj_parse.cu, load_obj(parser="gpu"), Pipeline(obj_parser="gpu")) returns
the host parser's arrays bit for bit and its errors word for word, and the pipeline's landmarks do not depend on
which parser read the scan."""
from pathlib import Path

import numpy as np
import pytest
import torch

from mvlm_b200 import synth
from mvlm_b200.io_obj import load_obj
from mvlm_b200.weights import seeded_state_dict

from test_obj_parse_cpu import CORPUS, _random_obj

pytestmark = pytest.mark.gpu


def same_as_host(path: Path):
    ref = load_obj(path, load_texture=False)
    got = load_obj(path, load_texture=False, parser="gpu")
    if isinstance(got.verts, torch.Tensor):
        got.geometry_ready.synchronize()
        verts, tris = got.verts.cpu().numpy(), got.tris.cpu().numpy()
        uvs = None if got.uvs is None else got.uvs.cpu().numpy()
        gpu = True
    else:
        verts, tris, uvs, gpu = got.verts, got.tris, got.uvs, False
    assert verts.dtype == np.float32 and tris.dtype == np.int32
    assert np.array_equal(verts.view(np.uint32), ref.verts.view(np.uint32))
    assert np.array_equal(tris, ref.tris)
    assert (uvs is None) == (ref.uvs is None)
    if uvs is not None:
        assert np.array_equal(uvs.view(np.uint32), ref.uvs.view(np.uint32))
    return gpu


def same_error(path: Path):
    with pytest.raises(ValueError) as host:
        load_obj(path, load_texture=False)
    with pytest.raises(ValueError) as gpu:
        load_obj(path, load_texture=False, parser="gpu")
    assert str(gpu.value) == str(host.value)
    return str(host.value)


def test_cpu_corpus_and_random_files(lib, tmp_path):
    n_gpu = 0
    cases = {name: text.encode() for name, text in CORPUS.items()}
    cases.update({f"r{seed}.obj": _random_obj(seed).encode() for seed in range(300)})
    for name, text in cases.items():
        p = tmp_path / name
        p.write_bytes(text)
        try:
            load_obj(p, load_texture=False)
        except ValueError:
            same_error(p)
            continue
        n_gpu += same_as_host(p)
    assert n_gpu > 100


def test_synthetic_scans(lib, tmp_path):
    v, uv, t = synth.face_mesh(grid=224, seed=1234)              # the 50k-vertex scan of the bench
    synth.write_obj(tmp_path / "scan.obj", v, uv, t, None)
    assert same_as_host(tmp_path / "scan.obj")
    v, uv, t = synth.face_mesh(grid=1001, seed=5)                 # config 4 size: 1M vertices, 2M triangles
    synth.write_obj(tmp_path / "big.obj", v, uv, t, None)
    assert same_as_host(tmp_path / "big.obj")
    synth.write_obj(tmp_path / "nouv.obj", v[:5000], None, t[t.max(1) < 5000], None)
    assert same_as_host(tmp_path / "nouv.obj")


def test_long_number_takes_the_host_parser(lib, tmp_path):
    p = tmp_path / "long.obj"
    p.write_text("v 1.00000005960464477539062500001 0 0\nv 1 0 0\nv 0 1 0\nvt 0 0\nf 1/1 2/1 3/1\n")
    assert not same_as_host(p)                                    # identical arrays, as numpy from the host parser


def test_errors(lib, tmp_path):
    cases = {
        "malformed_v.obj": "v 0 0 0\nv 1 x 0\nv 0 1 0\nf 1 2 3\n",
        "malformed_vt.obj": "v 0 0 0\nvt 1\nf 1 1 1\n",
        "malformed_f.obj": "v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3x\nf 1 2 9\n",
        "range.obj": "v 1e400 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3\n",
        "vertex_pos.obj": "v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3\nf 1 2 7\nf 1 2 8\n",
        "vertex_neg.obj": "v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 -4\nv 0 0 1\nf 1 2 -5\n",
        "vt_pos.obj": "v 0 0 0\nv 1 0 0\nv 0 1 0\nvt 0 0\nf 1/1 2/1 3/2\n",
        "vt_neg.obj": "v 0 0 0\nv 1 0 0\nv 0 1 0\nvt 0 0\nf 1/1 2/-3 3/1\n",
        "first_in_file.obj": "v 0 0 0\nv 1 0 0\nv 0 1 0\nvt 0 0\n" + "f 1 2 3\n" * 5000 + "f 1/1 2/5 9\nf 1 2 10\n",
        "no_points.obj": "# nothing\nvt 0 0\n",
        "empty.obj": "",
    }
    for name, text in cases.items():
        p = tmp_path / name
        p.write_text(text)
        msg = same_error(p)
        assert str(p) in msg
    assert "vt 5 of 1" in same_error(tmp_path / "first_in_file.obj")
    with pytest.raises(ValueError, match="does not exist"):
        load_obj(tmp_path / "missing.obj", parser="gpu")


@pytest.fixture(scope="module")
def scans(tmp_path_factory):
    d = tmp_path_factory.mktemp("scans")
    paths = []
    for i in range(3):
        v, uv, t = synth.face_mesh(grid=80 + 10 * i, seed=20 + i)
        paths.append(synth.write_obj(d / f"s{i}.obj", v, uv, t, synth.face_texture(256, seed=20 + i)))
    v, uv, t = synth.face_mesh(grid=90, seed=30)
    paths.append(synth.write_obj(d / "untextured.obj", v, None, t, None))
    return paths


@pytest.mark.parametrize("settings", [
    dict(seed=5), dict(seed=None), dict(seed=5, texture_decoder="nvjpeg"),
    dict(seed=5, pre_align={"align_center_of_mass": True, "rot_x": 10.0, "rot_y": -15.0, "rot_z": 5.0, "scale": 0.9}),
])
def test_pipeline_landmarks_do_not_depend_on_the_parser(lib, scans, tmp_path, settings):
    import mvlm

    kw = dict(n_views=8, weights=seeded_state_dict(73, "RGB+depth", 3), n_hypotheses=4, verbose=False,
              image_size=(64, 64), transforms=synth.random_view_transforms(8, seed=11), **settings)
    host = mvlm.pipeline.create_pipeline("dtu3d", **kw)
    gpu = mvlm.pipeline.create_pipeline("dtu3d", obj_parser="gpu", **kw)
    assert host.obj_parser == "host" and gpu.obj_parser == "gpu"
    seeded = settings["seed"] is not None
    for p in scans:
        if not seeded:
            np.random.seed(123)
        want = host.predict_one_file(p)
        if not seeded:
            np.random.seed(123)
        got = gpu.predict_one_file(p)
        assert np.array_equal(got, want), p
    if not seeded:
        np.random.seed(7)
    want = host.predict_files(scans, prefetch=3)
    if not seeded:
        np.random.seed(7)
    got = gpu.predict_files(scans, prefetch=3)
    assert all(np.array_equal(a, b) for a, b in zip(got, want))
    if seeded:
        out_h, out_g = tmp_path / "h", tmp_path / "g"
        rh = host.predict_folder(scans[0].parent, out_h)
        rg = gpu.predict_folder(scans[0].parent, out_g)
        assert rh.keys() == rg.keys() and all(np.array_equal(rh[k], rg[k]) for k in rh)
        assert sorted(f.read_bytes() for f in out_h.iterdir()) == sorted(f.read_bytes() for f in out_g.iterdir())
    with pytest.raises(ValueError, match="Unknown OBJ parser"):
        mvlm.pipeline.create_pipeline("dtu3d", obj_parser="nope", **kw)
