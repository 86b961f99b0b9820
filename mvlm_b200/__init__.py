"""mvlm_b200 -- B200-native multi-view 3D landmarking hot path behind the cvjena/mvlm Python API.

    import mvlm_b200 as mvlm            # or: import mvlm  (alias package at the repo root)
    dm = mvlm.pipeline.create_pipeline("dtu3d", n_views=100, weights=state_dict)
    landmarks = dm.predict_one_file(Path("scan.obj"))    # (73, 3) float64

All device work goes through libmvlm_b200.so (hand-written sm_100a CUDA, C-ABI in
include/mvlm_b200.h); there is no CPU fallback.
"""
__all__ = ["pipeline", "utils", "prediction", "LandmarkReport"]
__version__ = "0.1.0"


def __getattr__(name):
    # lazy: `import mvlm_b200.build` must work before the shared library exists
    if name == "LandmarkReport":
        from .report import LandmarkReport

        return LandmarkReport
    if name in __all__:
        import importlib

        return importlib.import_module(f"{__name__}.{name}")
    raise AttributeError(name)
