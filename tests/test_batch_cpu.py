"""Several scans per device pass, the parts that need no GPU: the pass planner, the multi-scan size queries and the
exported symbols."""
import ctypes as C

from mvlm_b200 import _lib
from mvlm_b200.pipeline import general_pipeline as gp


def test_pass_planner_sizes(monkeypatch):
    monkeypatch.setattr(gp, "PASS_PIXELS", 96 * 256 * 256)
    assert gp.scans_per_pass(8, 256, 256) == 12
    assert gp.scans_per_pass(12, 256, 256) == 8
    assert gp.scans_per_pass(8, 128, 128) == 48
    assert gp.scans_per_pass(8, 64, 64) == _lib.MAX_SCANS  # capped by the scan table of the kernels
    # the headline workload and anything larger: one scan per pass, as before batching
    assert gp.scans_per_pass(100, 256, 256) == 1
    assert gp.scans_per_pass(200, 512, 512) == 1
    assert gp.scans_per_pass(97, 256, 256) == 1
    # at least one scan even when one scan is over the budget, and no more views than one CNN plan may take
    assert gp.scans_per_pass(8, 256, 256, max_views=40) == 5
    assert gp.scans_per_pass(8, 256, 256, max_views=3) == 1
    monkeypatch.setattr(gp, "PASS_PIXELS", 0)
    assert gp.scans_per_pass(8, 256, 256) == 1


class _Predictor:
    def max_views_per_launch(self, v, h, w):
        return v


class _Renderer:
    def __init__(self, n_views, transforms=None):
        self.n_views, self.transforms, self.image_size = n_views, transforms, (256, 256)


class _Estimator:
    def __init__(self, seed):
        self.seed = seed


def _plan(n_views, seed, transforms=None):
    p = gp.Pipeline.__new__(gp.Pipeline)
    p.renderer_3d, p.estimator_3d, p.predictor_2d = _Renderer(n_views, transforms), _Estimator(seed), _Predictor()
    return p._scans_per_pass()


def test_pass_planner_rng_rule(monkeypatch):
    monkeypatch.setattr(gp, "PASS_PIXELS", 96 * 256 * 256)
    assert _plan(8, seed=1) == 12        # the preset views draw nothing
    assert _plan(8, seed=None) == 12     # only the consensus draws use the global RNG
    assert _plan(12, seed=1) == 8        # only the random views use it
    assert _plan(12, seed=None) == 1     # both: scan i's draws come before scan i+1's views
    assert _plan(12, seed=None, transforms=[[0] * 6] * 12) == 8  # given views draw nothing
    assert _plan(100, seed=1) == 1


def test_multiscan_size_queries(lib):
    # one scan: exactly the single-scan queries (the raster formula is pinned in test_host_cpu)
    assert lib.mvlm_raster_multiscan_workspace_bytes(1, 100, 256, 256, 50176) == lib.mvlm_raster_workspace_bytes(
        100, 256, 256, 50176)
    assert lib.mvlm_raster_multiscan_workspace_bytes(12, 8, 256, 256, 50176) == 96 * 256 * 256 * 8 + 96 * 50176 * 16
    # chunked over (scan, view) pairs beyond 256 MB of transformed vertices
    assert lib.mvlm_raster_multiscan_workspace_bytes(16, 8, 256, 256, 1002001) <= 128 * 256 * 256 * 8 + (256 << 20)
    for l, v, h in ((73, 8, 1), (84, 200, 16384)):
        assert lib.mvlm_consensus_multiscan_workspace_bytes(1, l, v, h) == lib.mvlm_consensus_workspace_bytes(l, v, h)
        assert lib.mvlm_consensus_multiscan_workspace_bytes(12, l, v, h) >= 12 * l * v * 16 * 8
    m = (_lib.SnapMesh * 1)()
    m[0].n_tris = 100000
    assert lib.mvlm_snap_to_meshes_workspace_bytes(m, 1, 73) == lib.mvlm_snap_grid_query_workspace_bytes(73, 100000)
    big = (_lib.SnapMesh * 3)()
    for e, nt in zip(big, (500, 100000, 2000)):
        e.n_tris = nt
    assert lib.mvlm_snap_to_meshes_workspace_bytes(big, 3, 73) >= lib.mvlm_snap_workspace_bytes(3 * 73, 100000)
    assert lib.mvlm_snap_to_meshes_workspace_bytes(big, 0, 73) == 0
    assert lib.mvlm_snap_to_meshes_workspace_bytes(big, _lib.MAX_SCANS + 1, 73) == 0


def test_multiscan_symbols_and_table_layout(lib):
    for name in ("mvlm_raster_multiscan", "mvlm_raster_multiscan_workspace_bytes", "mvlm_consensus_multiscan",
                 "mvlm_consensus_multiscan_workspace_bytes", "mvlm_snap_to_meshes", "mvlm_snap_to_meshes_workspace_bytes"):
        assert hasattr(lib, name)
    # ctypes mirrors of the C structs (x86-64 / aarch64 LP64 layout)
    assert C.sizeof(_lib.RasterScan) == 64
    assert _lib.RasterScan.tex.offset == 40
    assert C.sizeof(_lib.SnapMesh) == 40


def test_multiscan_rejects_bad_tables(lib):
    scans = (_lib.RasterScan * 1)()
    rc = lib.mvlm_raster_multiscan(scans, _lib.MAX_SCANS + 1, None, 8, 64, 64, 0, None, 0, None, None, None, None, None)
    assert rc != 0 and b"scans per pass" in lib.mvlm_last_error()
    rc = lib.mvlm_snap_to_meshes((_lib.SnapMesh * 1)(), 0, None, 73, None, 0, None, None, None)
    assert rc != 0 and b"scans per pass" in lib.mvlm_last_error()
