"""Host-side mirror of the reference's Estimator3D (src/mvlm/utils/estimator3d.py:18-285) on top
of the CUDA ray / consensus / snap kernels.  Same constructor, attributes and method signatures
(numpy in, numpy out); the fused pipeline calls the *_device variants to stay on the GPU.
"""
from __future__ import annotations

import numpy as np
import torch

from .. import ops
from ..io_obj import Mesh
from .render3d import rotation_matrices

__all__ = ["Estimator3D"]


class Estimator3D:
    def __init__(self, mode: str = "quantile", threshold_quantile: float = 0.5, threshold_absolute: float = 0.5,
                 n_hypotheses: int = 1, seed: int | None = None, device: str = "cuda"):
        self.mode = mode
        self.threshold_quantile = threshold_quantile
        self.threshold_absolute = threshold_absolute
        # extension of the reference's single draw (estimator3d.py:103-105): number of seeded hypotheses
        self.n_hypotheses = n_hypotheses
        self.seed = seed
        self.dist_thres = 10 * 10  # estimator3d.py:97
        self.device = torch.device(device)
        self.verbose = True

    # ---------------------------------------------------------------- rays (estimator3d.py:31-90)
    def estimate_landmark_lines(self, image_stack: np.ndarray, landmarks_stack: np.ndarray, transform_stack: np.ndarray):
        img_size = image_stack.shape[1]  # img_size == hm_size (:43-44)
        starts, ends = self.estimate_landmark_lines_device(
            torch.from_numpy(np.ascontiguousarray(landmarks_stack, dtype=np.float32)).to(self.device),
            transform_stack, img_size)
        return starts.cpu().numpy(), ends.cpu().numpy()

    def estimate_landmark_lines_device(self, peaks: torch.Tensor, transform_stack: np.ndarray, img_size: int, rot=None):
        """`rot`: optional (V,9) float64 device tensor of the view rotations (the renderer caches it)."""
        if rot is None:
            rot = torch.from_numpy(rotation_matrices(np.asarray(transform_stack)).reshape(-1, 9)).to(self.device)
        return ops.rays_from_peaks(peaks, rot, img_size)

    def seeded_draws_device(self, n_landmarks: int) -> torch.Tensor:
        key = (self.seed, self.n_hypotheses, n_landmarks)
        if getattr(self, "_draws_key", None) != key:
            self._draws = torch.from_numpy(self.seeded_draws(n_landmarks).view(np.int32)).to(self.device)
            self._draws_key = key
        return self._draws

    # ---------------------------------------------------------------- hypothesis tables
    def _filter_counts(self, values: np.ndarray) -> np.ndarray:
        if self.mode == "absolute":
            return (values > self.threshold_absolute).sum(1)
        if self.mode == "quantile":
            thr = np.array([np.quantile(values[i], self.threshold_quantile) for i in range(values.shape[0])])
            return (values > thr[:, None]).sum(1)
        raise ValueError(f"Unknown mode for line matching in Estimator: {self.mode}")

    def reference_draws(self, landmark_stack: np.ndarray) -> np.ndarray:
        """Replays the reference's RNG use: for every landmark with >= 3 filtered lines, in landmark
        order, `np.random.choice(range(n_lines), 8, replace=True)` on the GLOBAL numpy RNG
        (estimator3d.py:105), `n_hypotheses` times.  (L,H,8) uint32."""
        counts = self._filter_counts(np.asarray(landmark_stack)[:, :, 2])
        draws = np.zeros((len(counts), self.n_hypotheses, 8), dtype=np.uint32)
        for lm, n in enumerate(counts):
            if n >= 3:
                for h in range(self.n_hypotheses):
                    draws[lm, h] = np.random.choice(range(int(n)), 8, replace=True)
        return draws

    def seeded_draws(self, n_landmarks: int) -> np.ndarray:
        rs = np.random.RandomState(self.seed)
        return rs.randint(0, 2 ** 32, (n_landmarks, self.n_hypotheses, 8), dtype=np.uint64).astype(np.uint32)

    # ---------------------------------------------------------------- consensus (estimator3d.py:158-183)
    def estimate_landmarks_from_lines(self, landmark_stack, lines_s, lines_e, draws: np.ndarray | None = None):
        if self.mode not in ("absolute", "quantile"):
            raise ValueError(f"Unknown mode for line matching in Estimator: {self.mode}")
        landmark_stack = np.ascontiguousarray(landmark_stack, dtype=np.float32)
        if draws is None:
            draws = self.seeded_draws(landmark_stack.shape[0]) if self.seed is not None else self.reference_draws(landmark_stack)
        lm, err, nl = self.estimate_landmarks_from_lines_device(
            torch.from_numpy(landmark_stack).to(self.device),
            torch.from_numpy(np.ascontiguousarray(lines_s, dtype=np.float64)).to(self.device),
            torch.from_numpy(np.ascontiguousarray(lines_e, dtype=np.float64)).to(self.device),
            torch.from_numpy(np.ascontiguousarray(draws).view(np.int32)).to(self.device))
        nl = nl.cpu().numpy()
        if self.verbose:
            for lm_no in np.nonzero(nl < 3)[0]:
                print("Not enough points for good estimate of landmark lm_no", lm_no, nl[lm_no])
        err = err.cpu().numpy()
        return lm.cpu().numpy(), float(np.sum(err) / len(err))

    def estimate_landmarks_from_lines_device(self, peaks, starts, ends, draws, n_scans: int | None = None):
        """n_scans: peaks / starts / ends are the (L, S*V, 3) arrays of a pass of S scans (draws (L,H,8) shared or
        (S,L,H,8)); the results are then (S,L,3), (S,L), (S,L)."""
        kw = dict(mode=self.mode, threshold_quantile=self.threshold_quantile, threshold_absolute=self.threshold_absolute,
                  dist_thres=float(self.dist_thres))
        if n_scans is None:
            return ops.consensus(peaks, starts, ends, draws, **kw)
        return ops.consensus_multiscan(peaks, starts, ends, draws, n_scans, **kw)

    # ---------------------------------------------------------------- snap (estimator3d.py:252-285)
    def project_landmarks_to_surface(self, pd, landmarks):
        """`pd` is the mesh returned by the renderer (io_obj.Mesh or a renderer DeviceMesh)."""
        mesh = pd.mesh if hasattr(pd, "mesh") else pd
        if not isinstance(mesh, Mesh):
            raise TypeError("project_landmarks_to_surface expects the mesh returned by multiview_render")
        verts = pd.verts if hasattr(pd, "mesh") else torch.from_numpy(mesh.verts).to(self.device)
        tris = pd.tris if hasattr(pd, "mesh") else torch.from_numpy(mesh.tris).to(self.device)
        lm = torch.from_numpy(np.ascontiguousarray(landmarks, dtype=np.float64)).to(self.device)
        out, _ = ops.snap_to_mesh(verts, tris, lm, grid=pd.snap_grid() if hasattr(pd, "snap_grid") else "auto")
        return out.cpu().numpy()
