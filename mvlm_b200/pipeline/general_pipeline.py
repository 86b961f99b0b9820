"""Drop-in boundary: the reference's Pipeline (src/mvlm/pipeline/general_pipeline.py:39-146).

`predict_one_file(path)` keeps the reference's signature, error behaviour and stage prints.  When
the three components are the B200 ones (the default), the scan stays on the GPU from mesh upload
to the final (L,3) landmarks ("fused" path); if a user swapped in their own Predictor2D /
renderer / estimator, the reference's seam-by-seam numpy flow is used instead.
"""
from __future__ import annotations

__all__ = ["Pipeline"]

import abc
import dataclasses
import os
import time
from pathlib import Path

import numpy as np
import torch

from .. import _lib
from ..io_mesh import SUFFIXES, check_scan_file, check_scan_formats, check_scan_path, is_scan_file, load_mesh
from ..io_obj import Mesh, check_texture_source
from ..prediction.paulsenpredictor import PaulsenModel
from ..utils import Estimator3D, ObjRenderer3D, prealign

# Pixels of one device pass of the batch drivers.  The premise -- a plan of 8 views of 256^2 cannot fill the GPU and
# the views of several scans in one plan can -- is not measured yet (`tools/bench_batch.py --cnn --e2e` measures it),
# so the default is 0: one scan per pass, the work of one scan at a time.  MVLM_PASS_PIXELS sets a budget for
# measurements and tests; the candidate is about 96 views of 256^2 (12 scans of the 8-view preset per pass, while 100
# views of 256^2 stay one scan per pass), the issue's estimate, not a measured figure.
PASS_PIXELS = int(os.environ.get("MVLM_PASS_PIXELS", "0"))


def scans_per_pass(n_views: int, h: int, w: int, max_views: int | None = None) -> int:
    """Scans the batch drivers put into one device pass: as many as fit PASS_PIXELS (at least one, at most
    MVLM_MAX_SCANS), and no more views than one CNN plan may take (`max_views`)."""
    s = min(_lib.MAX_SCANS, max(1, PASS_PIXELS // (n_views * h * w)))
    if max_views is not None:
        s = min(s, max(1, max_views // n_views))
    return s


class _DeviceLock:
    """Re-entrant lock that also makes the pipeline's device the current CUDA device while it is held: every kernel
    of the library is launched on the current stream of the CURRENT device, so create_pipeline(device="cuda:1") must
    not depend on what the calling thread's current device happens to be."""

    def __init__(self, device: torch.device):
        import threading

        self._lock = threading.RLock()
        self._device = device
        self._guards = []

    def __enter__(self):
        self._lock.acquire()
        guard = torch.cuda.device(self._device) if self._device.type == "cuda" else None
        if guard is not None:
            guard.__enter__()
        self._guards.append(guard)
        return self

    def __exit__(self, *exc):
        guard = self._guards.pop()
        try:
            if guard is not None:
                guard.__exit__(*exc)
        finally:
            self._lock.release()
        return False


class TimeMixin:
    def __init__(self):
        self.start_time = time.time()
        self.end_time = None

    def tic(self):
        self.start_time = time.time()

    def toc(self):
        self.end_time = time.time()
        return self.end_time - self.start_time

    def toc_p(self):
        return self.p_time(self.toc())

    def p_time(self, t):
        return f"{t:08.6f} s"


class Pipeline(abc.ABC, TimeMixin):
    def __init__(self, render_image_stack: bool = False, offscreen: bool = True, n_views: int = 8,
                 render_image_folder: Path | None = None, visualize_rays: bool = False,
                 screenshot_folder: Path | None = None, *, image_size: tuple = (256, 256),
                 channel_mode: str = "RGB+depth", n_hypotheses: int = 1, seed: int | None = None,
                 transforms: np.ndarray | None = None, device: str = "cuda", verbose: bool = True,
                 texture_decoder: str = "pil", pre_align: dict | None = None, obj_parser: str = "host",
                 scan_formats: tuple = ("obj",), texture_source: str = "stem"):
        TimeMixin.__init__(self)
        self.render_image_stack = render_image_stack
        self.render_image_folder = render_image_folder
        self.n_views = n_views
        self.visualize_rays = visualize_rays  # accepted for compatibility; the VTK ray viewer is out of scope
        self.screenshot_folder = screenshot_folder
        self.verbose = verbose
        self.device = torch.device(device)
        # "pil": host decode (shared with the parity oracle); "nvjpeg": decode on the GPU into device memory
        self.texture_decoder = texture_decoder
        # "host": csrc/obj_loader.cu (numpy arrays); "gpu": csrc/obj_parse.cu, the same arrays bit for bit parsed on the
        # device (the host only reads the file).  Used by predict_one_file's fused path and predict_files /
        # predict_folder; the seam path (custom components, render_image_stack) and the view-split upload
        # (sharding.upload_mesh_sharded) take host arrays and keep the host parser.
        if obj_parser not in ("host", "gpu"):
            raise ValueError(f"Unknown OBJ parser: {obj_parser}")
        self.obj_parser = obj_parser
        # scan file formats predict_one_file / predict_files / predict_folder / the seam renderer accept: ("obj",) (the
        # default: the OBJ-only checks and messages) or any of "obj", "ply", "stl" (io_mesh; obj_parser then selects
        # the host or the device decoder for every format)
        self.scan_formats = check_scan_formats(scan_formats)
        # where an OBJ scan's texture comes from: "stem" (the reference's `<stem>.jpg` rule, the default) or "mtl" (its
        # MTL materials, several texture pages per scan; DESIGN.md 7g) in every entry point and the seam renderer
        self.texture_source = check_texture_source(texture_source)
        # legacy "pre-align" block (configs/*.json:59-84): {"align_center_of_mass", "rot_x", "rot_y", "rot_z", "scale"};
        # None / identity = off, see utils/prealign.py
        self.pre_align = None if prealign.is_identity(pre_align) else dict(pre_align)

        self.renderer_3d = ObjRenderer3D(image_size=image_size, offscreen=offscreen, n_views=n_views,
                                         channel_mode=channel_mode, device=device)
        self.renderer_3d.transforms = transforms
        self.renderer_3d.verbose = verbose
        self.renderer_3d.pre_align = self.pre_align
        self.renderer_3d.scan_formats = self.scan_formats
        self.renderer_3d.texture_source = self.texture_source
        self.estimator_3d = Estimator3D(n_hypotheses=n_hypotheses, seed=seed, device=device)
        self.estimator_3d.verbose = verbose
        # One pipeline object = one set of device buffers (renderer images, CNN workspace, CUDA graphs): calls from
        # several threads (the reference's FastAPI server shares one pipeline across its thread pool without a lock,
        # 3DMD_server.py:24-31) are serialised here.
        self._lock = _DeviceLock(self.device)
        self.predictor_2d = None  # assigned by the subclasses
        self.last_error = None    # "Landmarks [Error]" of the last scan (general_pipeline.py:109)

    def _print(self, *a):
        if self.verbose:
            print(*a)

    def get_lm_count(self) -> int:
        if self.predictor_2d is None:
            raise ValueError("Predictor2D is not initialized.")
        return self.predictor_2d.get_lm_count()

    # ------------------------------------------------------------------ general_pipeline.py:67-131
    def predict_one_file(self, file_name: Path, landmark_indices: list[int] | None = None,
                         view_indices: list[int] | None = None, clip_rays_to_mesh: bool = True):
        with self._lock:
            if self.predictor_2d is None:
                raise ValueError("Predictor2D is not initialized.")
            file_name = Path(file_name)
            full_s = time.time()
            if not file_name.exists():
                print(f"File {file_name} does not exist")
                return None
            fused = (isinstance(self.predictor_2d, PaulsenModel) and type(self.renderer_3d) is ObjRenderer3D
                     and type(self.estimator_3d) is Estimator3D and not self.render_image_stack
                     and self.predictor_2d.selection_method in ("simple", "moment"))
            if fused:
                r = self.renderer_3d
                check_scan_path(file_name, self.scan_formats)
                self.tic()
                mesh = load_mesh(file_name, texture_decoder=self.texture_decoder, device=self.device,
                                 parser=self.obj_parser, texture_source=self.texture_source)
                self._print("Render [1] - Setup time: ", self.toc_p())
                landmarks = self.predict_mesh(mesh)
                self._print("Landmarks 3D Total: ", self.p_time(time.time() - full_s))
                return landmarks
            return self._predict_seams(file_name, full_s)

    def predict_files(self, file_names, prefetch: int = 2) -> list:
        """Batch driver (the reference's main.py:50-62 loop is strictly serial): the native loader parses / decodes the
        next `prefetch` scans on background threads (the C parser and the JPEG decoder release the GIL) and the copies
        and launches of scan i+1 are enqueued while the GPU still works on scan i (see predict_meshes).
        Returns one (L,3) array (or None for a missing file) per input, in order."""
        with self._lock:
            from concurrent.futures import ThreadPoolExecutor

            if self.predictor_2d is None:
                raise ValueError("Predictor2D is not initialized.")
            files = [Path(f) for f in file_names]

            def load(f: Path):
                if not f.exists():
                    return None
                check_scan_path(f, self.scan_formats)
                # four parser threads per scan: with more, the loaders of `prefetch` scans oversubscribe the host and the
                # thread that feeds the GPU gets descheduled (measured on the 16-core box: 36 scans/s with 16, 51 with 4)
                return load_mesh(f, n_threads=4, texture_decoder=self.texture_decoder, device=self.device,
                                 parser=self.obj_parser, texture_source=self.texture_source)

            # `prefetch` loader threads, with the scans of a whole pass queued for them: the driver takes a pass's scans
            # at once and then waits for an earlier pass, the loaders keep working meanwhile
            ahead = max(prefetch, self._scans_per_pass())

            def meshes():
                with ThreadPoolExecutor(max_workers=max(1, prefetch)) as pool:
                    pending = [pool.submit(load, f) for f in files[:ahead]]
                    for i, f in enumerate(files):
                        mesh = pending.pop(0).result()
                        if i + ahead < len(files):
                            pending.append(pool.submit(load, files[i + ahead]))
                        if mesh is None:
                            print(f"File {f} does not exist")
                        yield mesh

            return self.predict_meshes(meshes())

    def predict_folder(self, path, out=None) -> dict:
        """The reference's batch loop (main.py:23-62) for this pipeline: every `*.obj` of a folder (sorted; with
        scan_formats, every file of an enabled format), or one file; landmarks are written as `<out>/<stem>_<pipeline name>.txt` with `np.savetxt(..., delimiter=",")`, files
        whose landmarks could not be predicted are skipped.  Returns {file: landmarks | None}."""
        path = Path(path)
        if not path.exists():
            raise FileNotFoundError(f"{path.as_posix()} does not exist.")
        default = self.scan_formats == ("obj",)
        if path.is_file():
            if default and path.suffix.lower() != ".obj":
                raise ValueError(f"{path.as_posix()} is not an .obj file.")
            if not default:
                check_scan_file(path, self.scan_formats)
            files, out_dir = [path], Path(out) if out is not None else path.parent
        elif default:
            files, out_dir = sorted(path.glob("*.obj")), Path(out) if out is not None else path
            if len(files) == 0:
                raise ValueError("Given folder does not contain any .obj files.")
        else:
            files = sorted(f for f in path.iterdir() if f.is_file() and is_scan_file(f, self.scan_formats))
            out_dir = Path(out) if out is not None else path
            if len(files) == 0:
                names = ", ".join(SUFFIXES[f] for f in self.scan_formats)
                raise ValueError(f"Given folder does not contain any {names} files.")
        out_dir.mkdir(parents=True, exist_ok=True)
        pname = getattr(self, "name", type(self).__name__.lower())
        results = dict(zip(files, self.predict_files(files)))
        for f, lm in results.items():
            if lm is None:
                print(f"Landmarks for {f} could not be predicted -> skipping file [{f.stem}] for pipeline {pname}")
                continue
            np.savetxt((out_dir / f"{f.stem}_{pname}.txt").as_posix(), lm, delimiter=",")
        return results

    def _scans_per_pass(self) -> int:
        """Pass size of the batch drivers (scans_per_pass for this pipeline's views).  One scan per pass when both the
        view list (random views) and the consensus draws (seed=None) come from the global numpy RNG: one scan at a time
        draws scan i's consensus draws, which depend on its peaks, before scan i+1's views, and a pass could not."""
        r, e = self.renderer_3d, self.estimator_3d
        if r.transforms is None and r.n_views != 8 and e.seed is None:
            return 1
        h, w = r.image_size[0], r.image_size[1]
        v = r.n_views if r.transforms is None else len(r.transforms)
        s = scans_per_pass(v, h, w)
        return s if s == 1 else scans_per_pass(v, h, w, self.predictor_2d.max_views_per_launch(s * v, h, w))

    def _enqueue_pass(self, meshes: list, transforms: np.ndarray | None = None, reserve_scans: int = 1):
        """Enqueues the whole hot path of the scans of one pass on the current stream WITHOUT waiting for it: host ->
        device copies of every scan, one raster sequence, one CNN plan over all views, rays, consensus and snap of all
        scans, device -> pinned-host copy of the (S, L*3 + 1) result.  Each scan's landmarks equal those of a pass of
        that scan alone.  `reserve_scans`: the pass size the caller plans (the persistent image and the result ring
        are sized for it, so that a shorter last pass allocates nothing).
        Returns (pinned host rows, CUDA event recorded after the copy, objects to keep alive until then)."""
        from .. import ops

        r, p, e = self.renderer_3d, self.predictor_2d, self.estimator_3d
        n = len(meshes)
        stacks, dmeshes, backs = [], [], []
        for mesh in meshes:  # views drawn scan by scan, in the order of one scan at a time
            t = np.asarray(r.generate_3d_transformations() if transforms is None else transforms)
            back = None
            if self.pre_align is not None:
                # the whole path runs on the pre-aligned scan; the snapped landmarks are mapped back in _finish_pass
                verts = mesh.verts
                if isinstance(verts, torch.Tensor):
                    # parser="gpu": prealign runs on numpy, so the vertices come back to the host (12 bytes per vertex,
                    # and this thread waits for the scan's parse); the aligned copy is uploaded like host-parsed vertices
                    mesh.geometry_ready.synchronize()
                    verts = verts.cpu().numpy()
                a, b = prealign.affine(verts, self.pre_align)
                mesh = dataclasses.replace(mesh, verts=prealign.apply(verts, a, b))
                back = (a, b)
            stacks.append(t)
            dmeshes.append(r.upload(mesh))
            backs.append(back)
        v = stacks[0].shape[0]
        out = r.render_pass(dmeshes, stacks, reserve_views=reserve_scans * v)
        all_views = np.concatenate(stacks)
        peaks = p.predict_landmarks_device(out["u8"])
        starts, ends = e.estimate_landmark_lines_device(peaks, all_views, r.image_size[0],
                                                        rot=r.rotations_device(all_views))
        if e.seed is not None:
            draws_d = e.seeded_draws_device(peaks.shape[0])  # one (L,H,8) table for every scan
        else:
            # reference RNG replay needs the per-landmark line counts -> one small D2H of the peak values (synchronises);
            # the draws are taken scan by scan, in the order of one scan at a time
            pk = peaks.cpu().numpy()
            draws = np.stack([e.reference_draws(pk[:, i * v:(i + 1) * v]) for i in range(n)])
            draws_d = torch.from_numpy(draws.view(np.int32)).to(self.device)
        lm, err, _ = e.estimate_landmarks_from_lines_device(peaks, starts, ends, draws_d, n_scans=n)
        snapped, _ = ops.snap_to_meshes([(d.verts, d.tris, d.snap_grid()) for d in dmeshes], lm)
        # the mean error per scan as one scan's (L,) sum, so last_error has the same bits in a pass of any size: one
        # (S,L) row reduction would not guarantee that, torch sizes its reduction blocks (and so the order of the sums
        # within a row) from the number of rows as well
        mean_err = torch.stack([x.sum() for x in err]).reshape(n, 1) / err.shape[1]
        result = torch.cat([snapped.reshape(n, -1), mean_err], dim=1)
        # ring of page-locked result buffers, allocated together on first use (cudaHostAlloc synchronises the device) and
        # sized for the planned pass: a shorter pass uses a prefix
        ring = self.__dict__.setdefault("_result_ring", [])
        if not ring or ring[0].shape[1] != result.shape[1] or ring[0].shape[0] < n:
            ring.clear()
            ring.extend(torch.empty((max(n, reserve_scans), result.shape[1]), dtype=result.dtype, pin_memory=True)
                        for _ in range(8))
        self._result_i = (getattr(self, "_result_i", -1) + 1) % len(ring)
        host = ring[self._result_i][:n]
        host.copy_(result, non_blocking=True)
        done = torch.cuda.Event()
        done.record()
        return host, done, (dmeshes, result, peaks, starts, ends, lm, backs)

    def _finish_pass(self, host: torch.Tensor, done, keep) -> list:
        """Waits for a pass of _enqueue_pass; returns its (L,3) landmarks per scan.  last_error and the prints follow
        the scans in order."""
        done.synchronize()
        rows = host.numpy().copy()
        out = []
        for row, back in zip(rows, keep[-1]):
            self.last_error = float(row[-1])
            self._print("Landmarks [Error]: ", f"{self.last_error:08.6f}", " mm")
            lm = row[:-1].reshape(-1, 3)
            out.append(lm if back is None else prealign.invert(lm, *back))
        return out

    def predict_mesh(self, mesh: Mesh, transforms: np.ndarray | None = None) -> np.ndarray:
        """Fused device path for an already loaded scan (host arrays in, (L,3) float64 out)."""
        with self._lock:
            return self._finish_pass(*self._enqueue_pass([mesh], transforms))[0]

    def predict_meshes(self, meshes, depth: int = 2) -> list:
        """Batch form of predict_mesh: same results, bit for bit, and the same use of the global numpy RNG.  Several
        scans share one device pass when PASS_PIXELS allows it (_scans_per_pass; one scan per pass by default), and up to
        `depth` passes are in flight -- the copies and launches of the next pass are enqueued (one stream, so buffers
        are reused in order) before the host waits for the landmarks of an earlier one, which keeps host-side latency
        off the GPU's critical path.  A None entry yields None."""
        with self._lock:
            assert depth < 8, "depth is bounded by the ring of result buffers"
            per_pass = self._scans_per_pass()
            self.renderer_3d.reserve_upload_slots(per_pass * (depth + 1))
            results, batch, where, inflight = [], [], [], []

            def finish(keep_in_flight: int):
                while len(inflight) > keep_in_flight:
                    handle, idx = inflight.pop(0)
                    for i, lm in zip(idx, self._finish_pass(*handle)):
                        results[i] = lm

            for mesh in meshes:
                results.append(None)
                if mesh is None:
                    continue
                batch.append(mesh)
                where.append(len(results) - 1)
                if len(batch) == per_pass:
                    inflight.append((self._enqueue_pass(batch, reserve_scans=per_pass), where))
                    batch, where = [], []
                    finish(depth)
            if batch:
                inflight.append((self._enqueue_pass(batch, reserve_scans=per_pass), where))
            finish(0)
            return results

    def _predict_seams(self, file_name: Path, full_s: float):
        self.tic()
        image_stack, transform_stack, pd = self.renderer_3d.multiview_render(file_name)
        self._print("Render [Total]: ", self.toc_p())
        if self.render_image_stack:
            self.visualize_image_stack(image_stack, file_name)
        self.tic()
        landmark_stack, valid = self.predictor_2d.predict_landmarks_from_images(image_stack)
        self._print("Prediction [Total]: ", self.toc_p())
        landmark_stack = landmark_stack[:, valid, :]
        transform_stack = transform_stack[valid]
        image_stack = image_stack[valid]
        self.tic()
        lines_s, lines_e = self.estimator_3d.estimate_landmark_lines(image_stack, landmark_stack, transform_stack)
        self._print("Landmarks [0] - From Heatmaps: ", self.toc_p())
        self.tic()
        landmarks, error = self.estimator_3d.estimate_landmarks_from_lines(landmark_stack, lines_s, lines_e)
        self._print("Landmarks [1] - From View Lines: ", self.toc_p())
        self.tic()
        landmarks = self.estimator_3d.project_landmarks_to_surface(pd, landmarks)
        if self.pre_align is not None:  # pd is the pre-aligned scan: back to the scan's own space (estimator3d.py:286)
            landmarks = prealign.invert(landmarks, *self.renderer_3d.last_pre_align)
        self._print("Landmarks [2] - Project to Surface: ", self.toc_p())
        self.last_error = error
        self._print("Landmarks [Error]: ", f"{error:08.6f}", " mm")
        self._print("Landmarks 3D Total: ", self.p_time(time.time() - full_s))
        return landmarks

    # general_pipeline.py:133-146
    def visualize_image_stack(self, image_stack: np.ndarray, file_name: Path):
        from PIL import Image

        save_folder = self.render_image_folder or file_name.parent
        if not Path(save_folder).exists():
            raise ValueError(f"Folder for --visualize-method flag [{save_folder}] does not exist.")
        for i in range(self.n_views):
            single_image = np.uint8(image_stack[i, :, :, 0:3] * 255)
            Image.fromarray(single_image).save(Path(save_folder) / f"{file_name.stem}_{i:02d}.png")
