"""Drop-in alias: `import mvlm` resolves to the B200-native implementation (mvlm_b200), so code
written against cvjena/mvlm (`mvlm.pipeline.create_pipeline(...)`, README.md:86-103) runs unchanged."""
import sys

import mvlm_b200
from mvlm_b200 import pipeline, prediction, utils  # noqa: F401
from mvlm_b200.report import LandmarkReport  # noqa: F401

__all__ = ["pipeline", "utils", "prediction", "LandmarkReport"]
for _n in ("pipeline", "utils", "prediction"):
    sys.modules[f"mvlm.{_n}"] = getattr(mvlm_b200, _n)
