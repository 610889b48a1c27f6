"""``meshrenderer_phong.Renderer`` (auto_pose/meshrenderer/meshrenderer_phong.py) on the GPU: the reference's OpenGL 4.5 phong
renderer restated as the CUDA rasteriser of csrc/render.cu (include/aae_b200.h: aae_render_frames / aae_render_crops).

``render`` keeps the reference's signature, return values and ``np.random`` draw order; ``render_frames_device`` and
``render_crops_device`` render whole batches of views of one model without leaving the device."""
import ctypes as C

import numpy as np
import torch

from .. import _lib
from . import camera
from .inout import load_ply, mesh_attributes

FIXED_LIGHT = (400.0, 400.0, 400.0)
DEFAULT_PHONG = {"ambient": 0.4, "diffuse": 0.8, "specular": 0.3}
WORKSPACE_BUDGET = 1 << 30          # bytes of visibility buffer per launch; larger batches are split


class RenderError(RuntimeError):
    pass


def fixed_light(phong=DEFAULT_PHONG):
    return np.array(FIXED_LIGHT + (phong["ambient"], phong["diffuse"], phong["specular"]), dtype=np.float64)


def random_light(phong=DEFAULT_PHONG, rng=np.random):
    """Renderer.render(random_light=True) (meshrenderer_phong.py:118-121): position 1000 * random(3), then diffuse, then
    specular jitter, in this draw order; the ambient weight stays fixed."""
    pos = 1000. * rng.random(3)
    d = phong["diffuse"] + 0.1 * (2 * rng.rand() - 1)
    s = phong["specular"] + 0.1 * (2 * rng.rand() - 1)
    return np.array([pos[0], pos[1], pos[2], phong["ambient"], d, s], dtype=np.float64)


class Renderer(object):
    """Renderer(models_cad_files, samples=1, vertex_tmp_store_folder='.', clamp=False, vertex_scale=1.0): one mesh per model
    file, selected by ``obj_id``.  Only ``samples == 1`` (ANTIALIASING: 1) is supported.  ``vertex_tmp_store_folder`` and
    ``clamp`` are accepted for compatibility (the reference caches the parsed models there; its clamped shader is disabled)."""

    def __init__(self, models_cad_files, samples=1, vertex_tmp_store_folder='.', clamp=False, vertex_scale=1.0, device=None):
        if int(samples) != 1:
            raise NotImplementedError("ANTIALIASING > 1 (multisampling) is not supported: sample positions are implementation-defined")
        if isinstance(models_cad_files, str):
            models_cad_files = [models_cad_files]
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else int(device))
        self._meshes = []
        self.n_vertices = []
        try:
            for path in models_cad_files:
                verts, faces = mesh_attributes(load_ply(path), vertex_scale)
                h = C.c_void_p()
                _lib.check(_lib.lib().aae_mesh_create(self.device.index, _lib.ptr(verts), len(verts), _lib.ptr(faces), len(faces),
                                                      C.byref(h)), "mesh create (%s)" % path)
                self._meshes.append(h)
                self.n_vertices.append(len(verts))
        except Exception:
            self.close()
            raise
        self._maps = {}

    # ------------------------------------------------------------------------------------------------ helpers
    def _mesh(self, obj_id):
        if not 0 <= int(obj_id) < len(self._meshes):
            raise IndexError("obj_id %d: the renderer holds %d models" % (obj_id, len(self._meshes)))
        return self._meshes[int(obj_id)]

    @staticmethod
    def _params(W, H, K, Rs, ts, near, far, lights_x, lights_y=None):
        n = len(Rs)
        ts = np.broadcast_to(np.asarray(ts, dtype=np.float64).reshape(-1, 3), (n, 3))
        lx = np.broadcast_to(np.asarray(lights_x, dtype=np.float64).reshape(-1, 6), (n, 6))
        ly = lx if lights_y is None else np.broadcast_to(np.asarray(lights_y, dtype=np.float64).reshape(-1, 6), (n, 6))
        proj = camera.projection_matrix(K, W, H, near, far).reshape(-1)
        P = np.zeros((n, _lib.RENDER_VIEW_FLOATS), dtype=np.float32)
        views, _ = camera.view_matrices_batch(np.asarray(Rs).reshape(n, 3, 3), ts)
        P[:, 0:16] = views.reshape(n, 16)
        P[:, 16:32] = proj
        P[:, 32:48] = camera.normal_matrices(views).reshape(n, 16)
        P[:, 48:54] = lx.astype(np.float32)
        P[:, 54:60] = ly.astype(np.float32)
        return P

    def _chunk(self, mesh, W, H):
        per_view = _lib.lib().aae_render_workspace_bytes(mesh, 1, int(W), int(H))
        return max(1, min(4096, WORKSPACE_BUDGET // per_view))

    def _nearest_maps(self, W, H, out_h, out_w):
        """INTER_NEAREST source index of every output column / row, for every source size (ae/augment.py:nearest_cells)"""
        from ..ae.augment import nearest_cells
        key = (W, H, out_h, out_w)
        if key not in self._maps:
            cols = np.zeros((W + 1, out_w), np.int32)
            rows = np.zeros((H + 1, out_h), np.int32)
            for s in range(1, W + 1):
                cols[s] = nearest_cells(out_w, s, dtype=np.int32)
            for s in range(1, H + 1):
                rows[s] = nearest_cells(out_h, s, dtype=np.int32)
            self._maps[key] = (torch.from_numpy(cols).to(self.device), torch.from_numpy(rows).to(self.device))
        return self._maps[key]

    @staticmethod
    def check_flags(flags, first=0):
        """Raises RenderError naming the views that could not be rendered (a vertex behind the near plane, nothing visible, or a
        crop window outside the frame)."""
        flags = np.asarray(flags)
        if not flags.any():
            return
        msgs = []
        for bit, what in ((_lib.RENDER_BEHIND_CAMERA, "a vertex at or behind the near plane"),
                          (_lib.RENDER_EMPTY, "nothing visible (are the vertices in mm?)"),
                          (_lib.RENDER_BAD_CROP, "the crop window lies outside the frame")):
            bad = np.nonzero(flags & bit)[0]
            if len(bad):
                msgs.append("%s in view(s) %s" % (what, (bad + first).tolist()[:20]))
        raise RenderError("; ".join(msgs))

    # ------------------------------------------------------------------------------------------------ device batches
    def render_frames_device(self, obj_id, W, H, K, Rs, ts, near, far, lights, check=True):
        """Full frames of len(Rs) views: (bgr uint8 [n,H,W,3], depth float32 [n,H,W], obj_bb int32 [n,4], flags int32 [n]),
        CUDA tensors.  lights: [6] or [n, 6] = (x, y, z, ambient, diffuse, specular).  Raises RenderError for views with a
        vertex behind the near plane unless check=False (then flags says which)."""
        mesh = self._mesh(obj_id)
        W, H, n = int(W), int(H), len(Rs)
        P = torch.from_numpy(self._params(W, H, K, Rs, ts, near, far, lights)).to(self.device)
        bgr = torch.empty((n, H, W, 3), dtype=torch.uint8, device=self.device)
        depth = torch.empty((n, H, W), dtype=torch.float32, device=self.device)
        bb = torch.empty((n, 4), dtype=torch.int32, device=self.device)
        flags = torch.empty((n,), dtype=torch.int32, device=self.device)
        step = self._chunk(mesh, W, H)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device)
            ws = torch.empty((_lib.lib().aae_render_workspace_bytes(mesh, min(step, n), W, H),), dtype=torch.uint8, device=self.device)
            for a in range(0, n, step):
                e = min(n, a + step)
                _lib.check(_lib.lib().aae_render_frames(mesh, _lib.ptr(P[a:e]), e - a, W, H, float(near), float(far), _lib.ptr(ws),
                                                        ws.numel(), _lib.ptr(bgr[a:e]), _lib.ptr(depth[a:e]), _lib.ptr(bb[a:e]),
                                                        _lib.ptr(flags[a:e]), C.c_void_p(stream.cuda_stream)), "render frames")
        if check:                      # an empty frame is a valid frame; a vertex behind the camera is not
            self.check_flags(flags.cpu().numpy() & _lib.RENDER_BEHIND_CAMERA)
        return bgr, depth, bb, flags

    def render_crops_device(self, obj_id, W, H, K, Rs, ts, near, far, lights_x, pad_factor, out_h, out_w, lights_y=None,
                            offsets=None, want_mask=False, check=True):
        """Square crops of len(Rs) views without materialising the frames: Dataset.extract_square_patch(frame, obj_bb (+
        offsets * (w, h)), pad_factor, INTER_NEAREST) of light x, and optionally the depth == 0 mask of that crop and the crop of
        light y around the unshifted box.  Returns a dict of CUDA tensors: x [n,out_h,out_w,3] uint8, mask (bool) and y when
        asked for, obj_bb int32 [n,4], flags int32 [n]."""
        mesh = self._mesh(obj_id)
        W, H, n = int(W), int(H), len(Rs)
        P = torch.from_numpy(self._params(W, H, K, Rs, ts, near, far, lights_x, lights_y)).to(self.device)
        cols, rows = self._nearest_maps(W, H, int(out_h), int(out_w))
        dev = self.device
        x = torch.empty((n, out_h, out_w, 3), dtype=torch.uint8, device=dev)
        mask = torch.empty((n, out_h, out_w), dtype=torch.uint8, device=dev) if want_mask else None
        y = torch.empty((n, out_h, out_w, 3), dtype=torch.uint8, device=dev) if lights_y is not None else None
        bb = torch.empty((n, 4), dtype=torch.int32, device=dev)
        flags = torch.empty((n,), dtype=torch.int32, device=dev)
        off = None
        if offsets is not None:
            off = torch.from_numpy(np.ascontiguousarray(np.asarray(offsets, dtype=np.float64).reshape(n, 2))).to(dev)
        step = self._chunk(mesh, W, H)
        sl = lambda t, a, e: None if t is None else _lib.ptr(t[a:e])   # noqa: E731
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev)
            ws = torch.empty((_lib.lib().aae_render_workspace_bytes(mesh, min(step, n), W, H),), dtype=torch.uint8, device=dev)
            for a in range(0, n, step):
                e = min(n, a + step)
                _lib.check(_lib.lib().aae_render_crops(mesh, _lib.ptr(P[a:e]), e - a, W, H, float(near), float(far), sl(off, a, e),
                                                       float(pad_factor), int(out_h), int(out_w), _lib.ptr(cols), _lib.ptr(rows),
                                                       _lib.ptr(ws), ws.numel(), _lib.ptr(x[a:e]), sl(mask, a, e), sl(y, a, e),
                                                       _lib.ptr(bb[a:e]), _lib.ptr(flags[a:e]), C.c_void_p(stream.cuda_stream)),
                           "render crops")
        if check:
            self.check_flags(flags.cpu().numpy())
        out = {"x": x, "obj_bb": bb, "flags": flags}
        if mask is not None:
            out["mask"] = mask.bool()
        if y is not None:
            out["y"] = y
        return out

    # ------------------------------------------------------------------------------------------------ reference surface
    def render(self, obj_id, W, H, K, R, t, near, far, random_light=False, phong=DEFAULT_PHONG):
        """(bgr uint8 [H,W,3], depth float32 [H,W]) as numpy, like the reference (meshrenderer_phong.py:98-165).  With
        random_light the light is drawn from np.random in the reference's order."""
        light = globals()["random_light"](phong) if random_light else fixed_light(phong)
        bgr, depth, _, _ = self.render_frames_device(obj_id, W, H, np.asarray(K), [np.asarray(R)], np.asarray(t), near, far, light)
        return bgr[0].cpu().numpy(), depth[0].cpu().numpy()

    def close(self):
        for h in getattr(self, "_meshes", []):
            _lib.lib().aae_mesh_destroy(h)
        self._meshes = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
