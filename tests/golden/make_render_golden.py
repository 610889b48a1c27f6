#!/usr/bin/env python
"""Generate tests/golden/render_golden.npz (and the ASCII mesh fixture render_mesh.ply) by running the REFERENCE's own renderer
host code.

Run in the build container only (needs /root/reference; the GPU box has no copy):

    python tests/golden/make_render_golden.py

OpenGL, progressbar and TensorFlow are not installable here, so they are replaced by stubs before the reference is imported
(the same technique as make_golden.py).  The gl_utils package __init__ (GLFW / EGL contexts) is bypassed: its camera and inout
modules are imported on their own.  ``glReadPixels`` answers with fixed synthetic frames, ``glUniform*`` calls are recorded.
Everything recorded below is computed by *reference* code:

* mesh              gl_utils/inout.py:load_ply on render_mesh.ply (ascii; the reference's binary branch cannot run under Python 3)
* camera            gl_utils/camera.py:Camera().realCamera(W, H, K, R, t, near, far).data for the template K and a few poses
* training stream   ae/dataset.py:render_training_images through the real meshrenderer_phong.Renderer.render: the rotation and
                    the light uniforms of every render call, and the resulting train_x / mask_x / train_y from the synthetic frames
* embedding batch   ae/dataset.py:render_embedding_image_batch from synthetic frames: batch and obj_bbs
"""
import os
import sys
import types

import numpy as np

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from make_golden import REF, install_stubs, template_dataset_kw  # noqa: E402

W, H = 720, 540
N_TRAIN = 8
GL_CONST = {"GL_BGR": 0x80E0, "GL_RED": 0x1903, "GL_UNSIGNED_BYTE": 0x1401, "GL_FLOAT": 0x1406}


def synthetic_frame(k):
    """frame k answered by glReadPixels: a textured rectangle of positive depth on a zero background"""
    rng = np.random.RandomState(1000 + k)
    depth = np.zeros((H, W), np.float32)
    bgr = np.zeros((H, W, 3), np.uint8)
    w, h = rng.randint(60, 260), rng.randint(60, 220)
    x, y = rng.randint(0, W - w), rng.randint(0, H - h)
    depth[y:y + h, x:x + w] = rng.uniform(600, 800, (h, w)).astype(np.float32)
    bgr[y:y + h, x:x + w] = rng.randint(1, 256, (h, w, 3))
    return bgr, depth


class GLStub(types.ModuleType):
    """OpenGL.GL: records uniforms; glReadPixels answers the colour and then the depth of synthetic_frame(k), k = 0, 1, ..."""

    def __init__(self):
        super().__init__("OpenGL.GL")
        self.__all__ = sorted(set(GL_CONST) | {"glClear", "glViewport", "glUniform3f", "glUniform1f", "glDrawElementsIndirect",
                                                "glNamedFramebufferReadBuffer", "glReadPixels", "GL_COLOR_BUFFER_BIT",
                                                "GL_DEPTH_BUFFER_BIT", "GL_STENCIL_BUFFER_BIT", "GL_TRIANGLES", "GL_UNSIGNED_INT",
                                                "GL_COLOR_ATTACHMENT0", "GL_COLOR_ATTACHMENT1", "ctypes"})
        self.uniforms = []
        self.reads = 0
        self.frame = 0
        import ctypes
        self.ctypes = ctypes
        for k, v in GL_CONST.items():
            setattr(self, k, v)

    def __getattr__(self, item):
        if item.startswith("__"):
            raise AttributeError(item)
        if item.startswith("GL_"):
            return 0
        return lambda *a, **k: None

    def glUniform3f(self, loc, x, y, z):
        self.uniforms.append((loc, np.float32(x), np.float32(y), np.float32(z)))

    def glUniform1f(self, loc, v):
        self.uniforms.append((loc, np.float32(v)))

    def glReadPixels(self, x, y, w, h, fmt, typ):
        bgr, depth = synthetic_frame(self.frame)
        self.reads += 1
        if fmt == GL_CONST["GL_BGR"]:
            return np.flipud(bgr).tobytes()
        self.frame += 1
        return np.flipud(depth).copy()


def import_reference(gl):
    install_stubs()
    ogl = types.ModuleType("OpenGL")
    ogl.GL = gl
    sys.modules["OpenGL"] = ogl
    sys.modules["OpenGL.GL"] = gl
    import auto_pose.meshrenderer as mr
    gu = types.ModuleType("auto_pose.meshrenderer.gl_utils")       # bypass the GLFW / EGL context imports of __init__
    gu.__path__ = [os.path.join(REF, "auto_pose", "meshrenderer", "gl_utils")]
    sys.modules[gu.__name__] = gu
    mr.gl_utils = gu
    from auto_pose.meshrenderer.gl_utils import camera, inout
    gu.Camera = camera.Camera
    from auto_pose.meshrenderer import meshrenderer_phong
    return camera, inout, meshrenderer_phong


def write_fixture(path):
    from oracle import render_oracle as RO
    RO.write_ply(path, RO.bumpy_sphere(1, seed=4))


def main():
    gl = GLStub()
    camera, inout, phong = import_reference(gl)
    out = {}
    # ---- 1. load_ply ---------------------------------------------------------------------------------------------
    ply = os.path.join(HERE, "render_mesh.ply")
    write_fixture(ply)
    m = inout.load_ply(ply)
    for k in ("pts", "normals", "colors", "faces"):
        out["ply_" + k] = np.asarray(m[k], np.float64)
    # ---- 2. camera matrices --------------------------------------------------------------------------------------
    cfg, kw = template_dataset_kw()
    K = np.array(eval(kw["k"])).reshape(3, 3)
    rng = np.random.RandomState(9)
    from auto_pose.ae.pysixd_stuff import transform
    poses, datas = [], []
    for i, (near, far) in enumerate([(10.0, 10000.0), (10.0, 10000.0), (1.0, 5000.0), (50.0, 3000.0)]):
        R = transform.random_rotation_matrix(rng.rand(3))[:3, :3]
        t = np.array([0, 0, 700.0]) if i < 2 else rng.uniform(-50, 50, 3) + [0, 0, 900.0]
        c = camera.Camera()
        c.realCamera(W, H, K, R, t, near, far)
        poses.append(np.concatenate([R.reshape(-1), t, [near, far]]))
        datas.append(c.data)
    out["cam_pose"], out["cam_data"] = np.array(poses), np.array(datas)
    # ---- 3. training images through the real Renderer.render ----------------------------------------------------
    from auto_pose.ae.dataset import Dataset
    kw = dict(kw)
    kw.update(noof_training_imgs=str(N_TRAIN), noof_bg_imgs="1", background_images_glob="/nonexistent/*.jpg")
    ds = Dataset("/tmp/unused", **kw)
    r = phong.Renderer.__new__(phong.Renderer)
    r._samples = 1
    r._fbo = types.SimpleNamespace(id=0)
    r._scene_buffer = types.SimpleNamespace(update=lambda data: calls.append(np.array(data)))
    calls = []
    ds._cache_renderer = r
    np.random.seed(1234)
    ds.render_training_images()
    out["train_scene_data"] = np.array(calls)                   # Camera data of every render call (x, y, x, y, ...)
    out["train_uniforms"] = np.array([u[1:] + (np.float32(0),) * (4 - len(u)) for u in gl.uniforms], np.float32)
    out["train_uniform_loc"] = np.array([u[0] for u in gl.uniforms])
    out["train_after"] = np.random.rand(4)                      # the state of np.random after the loop
    out["train_x"], out["mask_x"], out["train_y"] = ds.train_x, ds.mask_x, ds.train_y
    # ---- 4. embedding batch from synthetic frames ---------------------------------------------------------------
    gl.frame = 100
    kw2 = dict(kw)
    kw2.update(min_n_views="12", num_cyclo="2")
    ds2 = Dataset("/tmp/unused", **kw2)
    ds2._cache_renderer = r
    batch, bbs = ds2.render_embedding_image_batch(0, 4)
    out["emb_batch"], out["emb_obj_bbs"] = batch, bbs
    # ---- 5. the cache file name get_training_images writes for the template cfg --------------------------------------
    import tempfile
    tmp = tempfile.mkdtemp()
    cfg.set("Dataset", "NOOF_TRAINING_IMGS", str(N_TRAIN))
    ds3 = Dataset(tmp, **kw)
    ds3._cache_renderer = r
    ds3.get_training_images(tmp, cfg)
    out["cache_name"] = np.array(os.listdir(tmp)[0])
    import io
    buf = io.StringIO()
    cfg.write(buf)
    out["cache_cfg"] = np.array(buf.getvalue())
    np.savez_compressed(os.path.join(HERE, "render_golden.npz"), **out)
    print("wrote", sorted(out))


if __name__ == "__main__":
    main()
