"""The slice of auto_pose/ae/dataset.py the hot path touches: crop shape, the idx -> rotation table
(``viewsphere_for_embedding``, dataset.py:39-58, built on pysixd_stuff/view_sampler.py:19-188), ``embedding_size``
and the square-patch crop helper (dataset.py:354-373).  Rendering / augmentation (OpenGL, imgaug) are out of scope
(SURVEY.md section 2 rows 7, 11): ``render_embedding_image_batch`` and ``render_training_images`` render with the CUDA
renderer of augmentedautoencoder_b200/meshrenderer when MODEL_PATH is configured, or call a user-supplied renderer."""
import math

import numpy as np

from .utils import lazy_property

_GOLDEN = (1.0 + math.sqrt(5.0)) / 2.0
_ICO_VERTS = [(-1.0, _GOLDEN, 0.0), (1.0, _GOLDEN, 0.0), (-1.0, -_GOLDEN, 0.0), (1.0, -_GOLDEN, 0.0),
              (0.0, -1.0, _GOLDEN), (0.0, 1.0, _GOLDEN), (0.0, -1.0, -_GOLDEN), (0.0, 1.0, -_GOLDEN),
              (_GOLDEN, 0.0, -1.0), (_GOLDEN, 0.0, 1.0), (-_GOLDEN, 0.0, -1.0), (-_GOLDEN, 0.0, 1.0)]
_ICO_FACES = [(0, 11, 5), (0, 5, 1), (0, 1, 7), (0, 7, 10), (0, 10, 11), (1, 5, 9), (5, 11, 4), (11, 10, 2), (10, 7, 6),
              (7, 1, 8), (3, 9, 4), (3, 4, 2), (3, 2, 6), (3, 6, 8), (3, 8, 9), (4, 9, 5), (2, 4, 11), (6, 2, 10),
              (8, 6, 7), (9, 8, 1)]


def icosphere_points(min_n_pts, radius=1.0):
    """Hinterstoisser view sphere: subdivide an icosahedron until it has >= min_n_pts vertices, push the vertices
    to the sphere and order them ring by ring from the top pole, each ring sorted by azimuth.  The vertex numbering,
    midpoint arithmetic and ring construction reproduce view_sampler.hinter_sampling exactly (checked bit-for-bit
    against tests/golden/viewsphere_*.npz)."""
    verts = [list(v) for v in _ICO_VERTS]
    faces = list(_ICO_FACES)
    while len(verts) < min_n_pts:
        midpoint = {}
        refined = []
        for tri in faces:
            mids = []
            for a, b in ((tri[0], tri[1]), (tri[1], tri[2]), (tri[2], tri[0])):
                key = (a, b) if a < b else (b, a)
                if key not in midpoint:
                    midpoint[key] = len(verts)
                    verts.append((0.5 * (np.array(verts[key[0]]) + np.array(verts[key[1]]))).tolist())
                mids.append(midpoint[key])
            v0, v1, v2 = tri
            m01, m12, m20 = mids
            refined += [(v0, m01, m20), (m01, v1, m12), (m01, m12, m20), (m20, m12, v2)]
        faces = refined
    pts = np.array(verts)
    pts *= np.reshape(radius / np.linalg.norm(pts, axis=1), (pts.shape[0], 1))
    neighbours = {}
    for tri in faces:
        for i in range(3):
            neighbours.setdefault(tri[i], set()).update((tri[(i + 1) % 3], tri[(i + 2) % 3]))
    two_pi = 2.0 * math.pi
    azimuth = [(math.atan2(p[1], p[0]) + two_pi) % two_pi for p in pts]
    visited = [False] * len(pts)
    ring = [int(np.argmax(pts[:, 2]))]
    order = []
    while len(order) != len(pts):
        ring = sorted(ring, key=azimuth.__getitem__)
        reach = []
        for v in ring:
            order.append(v)
            visited[v] = True
            reach += [i for i in neighbours[v]]
        ring = [i for i in set(reach) if not visited[i]]  # set iteration order decides azimuth ties, as upstream
    return pts[np.array(order), :]


def look_at_rotations(pts):
    """Camera rotation for every view point: the camera looks at the origin with world +z up (OpenGL look-at), then a
    180 degree flip about x converts to the OpenCV convention (view_sampler.sample_views, view_sampler.py:160-181)."""
    c, s = math.cos(math.pi), math.sin(math.pi)
    flip = np.array([[1.0, 0.0, 0.0], [0.0, c, -s], [0.0, s, c]])
    up = np.array([0.0, 0.0, 1.0])
    out = np.empty((len(pts), 3, 3))
    for i, pt in enumerate(pts):
        fwd = -np.array(pt)
        fwd /= np.linalg.norm(fwd)
        side = np.cross(fwd, up)
        if np.count_nonzero(side) == 0:
            side = np.array([1.0, 0.0, 0.0])
        side /= np.linalg.norm(side)
        upv = np.cross(side, fwd)
        out[i] = flip.dot(np.array([[side[0], side[1], side[2]], [upv[0], upv[1], upv[2]], [-fwd[0], -fwd[1], -fwd[2]]]))
    return out


def viewsphere_rotations(min_n_views, num_cyclo, radius):
    views = look_at_rotations(icosphere_points(min_n_views, radius=radius))
    rs = np.empty((len(views) * num_cyclo, 3, 3))
    angles = np.linspace(0, 2.0 * np.pi, num_cyclo)  # both end points included -> first and last in-plane step coincide
    i = 0
    for view in views:
        for cyclo in angles:
            rot_z = np.array([[np.cos(-cyclo), -np.sin(-cyclo), 0], [np.sin(-cyclo), np.cos(-cyclo), 0], [0, 0, 1]])
            rs[i] = rot_z.dot(view)
            i += 1
    return rs


def calc_2d_bbox(covered, im_size):
    """view_sampler.calc_2d_bbox (ae/pysixd_stuff/view_sampler.py:10-15) of the covered pixels: min / max +-1 pixel, clamped to
    (W - 1, H - 1); [x, y, w, h]"""
    ys, xs = np.nonzero(covered)
    x0, y0 = max(xs.min() - 1, 0), max(ys.min() - 1, 0)
    x1, y1 = min(xs.max() + 1, im_size[0] - 1), min(ys.max() + 1, im_size[1] - 1)
    return [x0, y0, x1 - x0, y1 - y0]


def random_rotation_matrix():
    """pysixd transform.random_rotation_matrix (ae/pysixd_stuff/transform.py:1463-1503): a uniform random unit quaternion from
    np.random.rand(3), as a homogeneous 4x4 rotation"""
    rand = np.random.rand(3)
    r1, r2 = np.sqrt(1.0 - rand[0]), np.sqrt(rand[0])
    t1, t2 = math.pi * 2.0 * rand[1], math.pi * 2.0 * rand[2]
    q = np.array([np.cos(t2) * r2, np.sin(t1) * r1, np.cos(t1) * r1, np.sin(t2) * r2], dtype=np.float64)
    n = np.dot(q, q)
    if n < np.finfo(float).eps * 4.0:
        return np.identity(4)
    q *= math.sqrt(2.0 / n)
    q = np.outer(q, q)
    return np.array([[1.0 - q[2, 2] - q[3, 3], q[1, 2] - q[3, 0], q[1, 3] + q[2, 0], 0.0],
                     [q[1, 2] + q[3, 0], 1.0 - q[1, 1] - q[3, 3], q[2, 3] - q[1, 0], 0.0],
                     [q[1, 3] - q[2, 0], q[2, 3] + q[1, 0], 1.0 - q[1, 1] - q[2, 2], 0.0],
                     [0.0, 0.0, 0.0, 1.0]])


class Dataset(object):
    """Constructor signature of auto_pose/ae/dataset.py:16-36 (``Dataset(dataset_path, **kw)`` with the lower-cased
    cfg keys).  Only what the encoder / codebook path needs is kept."""

    def __init__(self, dataset_path=None, renderer=None, **kw):
        self.shape = (int(kw.get("h", 128)), int(kw.get("w", 128)), int(kw.get("c", 3)))
        self.dataset_path = dataset_path
        self._kw = dict(kw)
        self._kw.setdefault("num_cyclo", 36)
        self._kw.setdefault("min_n_views", 2562)
        self._kw.setdefault("radius", 700)
        self._renderer = renderer

    @lazy_property
    def viewsphere_for_embedding(self):
        kw = self._kw
        return viewsphere_rotations(int(kw["min_n_views"]), int(kw["num_cyclo"]), float(kw["radius"]))

    @property
    def embedding_size(self):
        return len(self.viewsphere_for_embedding)

    # ------------------------------------------------------------------------------------------------ rendering
    @property
    def has_gpu_renderer(self):
        """True when views are rendered by the CUDA renderer: no renderer callable was passed and a MODEL_PATH is configured"""
        return self._renderer is None and bool(self._kw.get("model_path"))

    @lazy_property
    def renderer(self):
        """meshrenderer_phong.Renderer of MODEL_PATH (dataset.py:61-80), built on first use"""
        kw = self._kw
        model = str(kw.get("model", "reconst"))
        if model == "cad":
            raise NotImplementedError("MODEL: cad (pyassimp meshes, recalculated normals) is not supported; use MODEL: reconst")
        if model != "reconst":
            raise ValueError("MODEL must be reconst or cad, got %r" % model)
        from ..meshrenderer.meshrenderer_phong import Renderer
        return Renderer([kw["model_path"]], int(kw.get("antialiasing", 1)), self.dataset_path, float(kw.get("vertex_scale", 1.0)))

    def _render_setup(self):
        kw = self._kw
        if self.shape[2] != 3:
            raise NotImplementedError("C = 1 (grayscale) rendering is not supported")
        W, H = eval(str(kw.get("render_dims", "(720, 540)")))
        K = np.array(eval(str(kw.get("k", "[1075.65, 0, 720/2, 0, 1073.90, 540/2, 0, 0, 1]")))).reshape(3, 3)
        t = np.array([0, 0, float(kw["radius"])])
        return int(W), int(H), K, t, float(kw.get("clip_near", 10)), float(kw.get("clip_far", 10000)), float(kw.get("pad_factor", 1.2))

    def embedding_crops_device(self, start, end):
        """uint8 crops [n,H,W,3] and obj_bbs int32 [n,4] of codebook rows start..end as CUDA tensors: the views are rendered with
        the fixed light and cropped without leaving the device (dataset.py:308-352 without the / 255)."""
        from ..meshrenderer.meshrenderer_phong import fixed_light
        W, H, K, t, near, far, pad = self._render_setup()
        out = self.renderer.render_crops_device(0, W, H, K, self.viewsphere_for_embedding[start:end], t, near, far, fixed_light(), pad,
                                                self.shape[0], self.shape[1])
        return out["x"], out["obj_bb"]

    def render_embedding_image_batch(self, start, end):
        """(batch [n,H,W,C] float in [0,1], obj_bbs [n,4]) for codebook rows start..end (dataset.py:308-352).  Renders on the GPU
        when MODEL_PATH is configured, else through a renderer callable ``renderer(R) -> (bgr uint8 image, depth)``."""
        if self._renderer is None and self.has_gpu_renderer:
            crops, bbs = self.embedding_crops_device(start, end)
            return crops.cpu().numpy() / 255., bbs.cpu().numpy().astype(np.float64)
        if self._renderer is None:
            raise NotImplementedError("no renderer attached: configure model_path, pass renderer=callable(R)->(bgr, depth) to "
                                      "Dataset, or build the codebook with Codebook.update_embedding_from_crops")
        import cv2
        kw = self._kw
        h, w = self.shape[:2]
        pad_factor = float(kw.get("pad_factor", 1.2))
        batch = np.empty((end - start,) + self.shape)
        obj_bbs = np.empty((end - start, 4))
        for i, R in enumerate(self.viewsphere_for_embedding[start:end]):
            bgr, depth = self._renderer(R)
            obj_bbs[i] = calc_2d_bbox(depth > 0, (depth.shape[1], depth.shape[0]))
            crop = self.extract_square_patch(bgr, obj_bbs[i], pad_factor, resize=(w, h), interpolation=cv2.INTER_NEAREST)
            batch[i] = crop / 255.
        return batch, obj_bbs

    def extract_square_patch(self, scene_img, bb_xywh, pad_factor, resize=(128, 128), interpolation=None, black_borders=False):
        """Square crop around a bbox, clipped to the image, optional blackening outside the bbox (dataset.py:354-373)."""
        import cv2
        if interpolation is None:
            interpolation = cv2.INTER_NEAREST
        x, y, w, h = np.array(bb_xywh).astype(np.int32)
        size = int(np.maximum(h, w) * pad_factor)
        left = int(np.maximum(x + w / 2 - size / 2, 0))
        right = int(np.minimum(x + w / 2 + size / 2, scene_img.shape[1]))
        top = int(np.maximum(y + h / 2 - size / 2, 0))
        bottom = int(np.minimum(y + h / 2 + size / 2, scene_img.shape[0]))
        crop = scene_img[top:bottom, left:right].copy()
        if black_borders:
            crop[:(y - top), :] = 0
            crop[(y + h - top):, :] = 0
            crop[:, :(x - left)] = 0
            crop[:, (x + w - left):] = 0
        return cv2.resize(crop, resize, interpolation=interpolation)

    def training_draws(self, n):
        """The np.random draws of n training images in the reference's order (dataset.py:243-282): per image the rotation
        (random_rotation_matrix: rand(3)), the random light of x (random(3), rand, rand), then the two bbox offsets
        (uniform(-MAX_REL_OFFSET, MAX_REL_OFFSET) each).  Returns (Rs [n,3,3], lights [n,6], offsets [n,2])."""
        from ..meshrenderer.meshrenderer_phong import random_light
        m = float(self._kw.get("max_rel_offset", 0.20))
        Rs, lights, offs = np.empty((n, 3, 3)), np.empty((n, 6)), np.empty((n, 2))
        for i in range(n):
            Rs[i] = random_rotation_matrix()[:3, :3]
            lights[i] = random_light()
            offs[i, 0] = np.random.uniform(-m, m)
            offs[i, 1] = np.random.uniform(-m, m)
        return Rs, lights, offs

    def training_images_from_frames(self, bgr_x, depth_x, bgr_y, depth_y, offsets):
        """(train_x, mask_x, train_y) composed on the host from full frames, as the reference's loop does after its two render
        calls (dataset.py:271-303): bbox of depth x, crop of bgr x and depth x at the bbox shifted by offsets * (w, h), mask =
        depth crop == 0, crop of bgr y at the bbox of depth y.  render_training_images computes the same on the device."""
        import cv2
        h, w = self.shape[:2]
        pad = float(self._kw.get("pad_factor", 1.2))
        xs, ms, ys = [], [], []
        for i in range(len(bgr_x)):
            size = (depth_x[i].shape[1], depth_x[i].shape[0])
            bb = np.array(calc_2d_bbox(depth_x[i] > 0, size))
            off = bb + np.array([offsets[i][0] * bb[2], offsets[i][1] * bb[3], 0, 0])
            xs.append(self.extract_square_patch(bgr_x[i], off, pad, resize=(w, h), interpolation=cv2.INTER_NEAREST).astype(np.uint8))
            ms.append(self.extract_square_patch(depth_x[i], off, pad, resize=(w, h), interpolation=cv2.INTER_NEAREST) == 0.)
            bb_y = calc_2d_bbox(depth_y[i] > 0, size)
            ys.append(self.extract_square_patch(bgr_y[i], bb_y, pad, resize=(w, h), interpolation=cv2.INTER_NEAREST).astype(np.uint8))
        return np.array(xs), np.array(ms), np.array(ys)

    def render_training_images(self, batch=4096):
        """train_x (uint8), mask_x (bool) and train_y (uint8) of NOOF_TRAINING_IMGS images (dataset.py:219-306): x with a random
        light cropped around its bbox shifted by the random offset, its background mask, y with the fixed light around the
        unshifted bbox.  One render call per batch produces all three without materialising a frame."""
        from ..meshrenderer.meshrenderer_phong import fixed_light
        n = int(self._kw["noof_training_imgs"])
        W, H, K, t, near, far, pad = self._render_setup()
        h, w = self.shape[:2]
        Rs, lights, offs = self.training_draws(n)
        self.train_x = np.empty((n,) + self.shape, np.uint8)
        self.mask_x = np.empty((n, h, w), bool)
        self.train_y = np.empty((n,) + self.shape, np.uint8)
        for a in range(0, n, batch):
            e = min(n, a + batch)
            out = self.renderer.render_crops_device(0, W, H, K, Rs[a:e], t, near, far, lights[a:e], pad, h, w, lights_y=fixed_light(),
                                                    offsets=offs[a:e], want_mask=True, check=False)
            self.renderer.check_flags(out["flags"].cpu().numpy(), first=a)
            self.train_x[a:e] = out["x"].cpu().numpy()
            self.mask_x[a:e] = out["mask"].cpu().numpy()
            self.train_y[a:e] = out["y"].cpu().numpy()
        self.noof_training_imgs = n

    def get_training_images(self, dataset_path, args):
        """Load the cached training set for this cfg or render and cache it (dataset.py:83-97).  The cache file name is the md5
        of the [Dataset] and [Paths] items, as the reference names it, so caches written by either side load in the other."""
        import hashlib
        import os
        digest = hashlib.md5((str(args.items("Dataset") + args.items("Paths"))).encode("utf-8")).hexdigest()
        name = os.path.join(dataset_path, digest + ".npz")
        if os.path.exists(name):
            self.load_training_images(name)
        else:
            self.render_training_images()
            np.savez(name, train_x=self.train_x, mask_x=self.mask_x, train_y=self.train_y)
        self.noof_obj_pixels = np.count_nonzero(self.mask_x == 0, axis=(1, 2))
        return name

    # ------------------------------------------------------------------------------------------------ training batches
    def load_training_images(self, path, bg_path=None):
        """The cache the reference writes after rendering (``np.savez(current_file_name, train_x=, mask_x=, train_y=)``,
        dataset.py:101-113) and, optionally, the background image stack (``.npy``, dataset.py:229-255)."""
        data = np.load(path)
        self.train_x, self.mask_x, self.train_y = data["train_x"].astype(np.uint8), data["mask_x"], data["train_y"].astype(np.uint8)
        self.noof_training_imgs = len(self.train_x)
        if bg_path is not None:
            self.bg_imgs = np.load(bg_path).astype(np.uint8)
            self.noof_bg_imgs = len(self.bg_imgs)

    @lazy_property
    def _aug(self):
        from .augment import Augmenter
        code = self._kw.get("code")
        if code is None:
            raise NotImplementedError("no [Augmentation] CODE in the dataset arguments")
        return Augmenter(code, self.shape, seed=self._kw.get("seed"))

    def batch_device(self, batch_size, device=None):
        """Dataset.batch (dataset.py:456-495) with the image work on the GPU: draws the rendering / background indices like the
        reference, uploads the uint8 images once and returns (x, y) float32 CUDA tensors in [0, 1]."""
        import torch
        for name in ("train_x", "mask_x", "train_y", "bg_imgs"):
            if not hasattr(self, name):
                raise RuntimeError("Dataset.%s is not loaded (load_training_images / set the arrays)" % name)
        if eval(str(self._kw.get("realistic_occlusion", "False"))) or eval(str(self._kw.get("square_occlusion", "False"))):
            raise NotImplementedError("REALISTIC_OCCLUSION / SQUARE_OCCLUSION are off in the template cfg and not supported")
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else device
        idx = np.random.choice(len(self.train_x), batch_size, replace=False)
        idx_bg = np.random.choice(len(self.bg_imgs), batch_size, replace=False)
        x = torch.from_numpy(self.train_x[idx]).to(dev, non_blocking=True)
        m = torch.from_numpy(np.ascontiguousarray(self.mask_x[idx]).astype(np.uint8)).to(dev, non_blocking=True)
        bg = torch.from_numpy(self.bg_imgs[idx_bg]).to(dev, non_blocking=True)
        y = torch.from_numpy(self.train_y[idx]).to(dev, non_blocking=True)
        xf = self._aug.augment_device(x, m, bg)
        return xf, y.to(torch.float32) / 255.0

    def batch(self, batch_size):
        """numpy (batch_x, batch_y) like the reference's ``Dataset.batch``."""
        x, y = self.batch_device(batch_size)
        return x.cpu().numpy(), y.cpu().numpy()
