"""CPU tests of the renderer's host side: PLY reading, camera matrices, the training draw order, and known answers of the
numpy restatement (oracle/render_oracle.py) that the GPU renderer is compared against bit for bit."""
import numpy as np
import pytest

from augmentedautoencoder_b200.meshrenderer import camera
from augmentedautoencoder_b200.meshrenderer.inout import load_ply, mesh_attributes
from oracle import render_oracle as RO


@pytest.fixture(scope="module")
def sphere():
    return RO.bumpy_sphere(2, seed=1)


def test_ascii_and_binary_ply_give_identical_arrays(tmp_path, sphere):
    a = load_ply(RO.write_ply(str(tmp_path / "a.ply"), sphere))
    b = load_ply(RO.write_ply(str(tmp_path / "b.ply"), sphere, binary=True))
    for k in ("pts", "normals", "colors", "faces"):
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(a["pts"], sphere["pts"].astype(np.float32).astype(np.float64))
    assert np.array_equal(a["faces"], sphere["faces"])
    assert np.array_equal(a["colors"], sphere["colors"])


def test_mesh_attributes_follow_the_reference_upload(tmp_path, sphere):
    m = dict(sphere)
    del m["colors"]
    verts, faces = mesh_attributes(load_ply(RO.write_ply(str(tmp_path / "n.ply"), m)), vertex_scale=2.0)
    assert verts.dtype == np.float32 and verts.shape == (len(m["pts"]), 9) and faces.dtype == np.int32
    assert np.all(verts[:, 6:] == np.float32(160.0) / np.float32(255.0))
    assert np.array_equal(verts[:, :3], m["pts"].astype(np.float32) * 2.0)


def test_load_ply_of_a_large_model_is_vectorised(tmp_path):
    import time
    path = RO.write_ply(str(tmp_path / "big.ply"), RO.bumpy_sphere(6), binary=True)
    t0 = time.time()
    m = load_ply(path)
    assert len(m["faces"]) == 81920 and time.time() - t0 < 1.0


@pytest.mark.parametrize("case", ["quad", "no_normals", "truncated_ascii", "truncated_binary", "bad_format"])
def test_malformed_ply_raises_value_error(tmp_path, sphere, case):
    p = str(tmp_path / "x.ply")
    if case == "quad":
        open(p, "w").write("ply\nformat ascii 1.0\nelement vertex 4\nproperty float x\nproperty float y\nproperty float z\n"
                           "property float nx\nproperty float ny\nproperty float nz\nelement face 1\n"
                           "property list uchar int vertex_indices\nend_header\n" + "0 0 0 0 0 1\n" * 4 + "4 0 1 2 3\n")
    elif case == "no_normals":
        open(p, "w").write("ply\nformat ascii 1.0\nelement vertex 3\nproperty float x\nproperty float y\nproperty float z\n"
                           "element face 1\nproperty list uchar int vertex_indices\nend_header\n" + "0 0 0\n" * 3 + "3 0 1 2\n")
    elif case == "truncated_ascii":
        RO.write_ply(p, sphere)
        data = open(p, "rb").read()
        open(p, "wb").write(data[:len(data) // 2])
    elif case == "truncated_binary":
        RO.write_ply(p, sphere, binary=True)
        data = open(p, "rb").read()
        open(p, "wb").write(data[:-5])
    else:
        RO.write_ply(p, sphere)
        data = open(p, "rb").read().replace(b"format ascii", b"format binary_big_endian")
        open(p, "wb").write(data)
    with pytest.raises(ValueError):
        load_ply(p)


def test_camera_projects_pixel_centres_like_opencv():
    """pixel (c, r) of the read-back image samples u = K X / Z at (c + 0.5, r + 0.5)"""
    K = RO.TEMPLATE_K
    R = np.eye(3)
    t = np.array([0.0, 0.0, 700.0])
    view, _ = camera.view_matrices(R, t)
    proj = camera.projection_matrix(K, 720, 540, 10.0, 10000.0)
    pts = np.array([[10.0, -20.0, 5.0], [-50.0, 30.0, -40.0]], np.float32)
    X, Y, zw, cw, camz = RO.project(view, proj, pts, 720, 540)
    Xc = pts.astype(np.float64) + t
    u = K[0, 0] * Xc[:, 0] / Xc[:, 2] + K[0, 2]
    v = K[1, 1] * Xc[:, 1] / Xc[:, 2] + K[1, 2]
    assert np.allclose(X / 256.0, u, atol=2e-2) and np.allclose(Y / 256.0, v, atol=2e-2)
    assert np.allclose(camz, Xc[:, 2], rtol=1e-6)
    d = camera.camera_data(720, 540, K, R, t, 10.0, 10000.0)
    assert d.dtype == np.float32 and d.shape == (35,)
    assert np.allclose(d[32:], [0, 0, -700], atol=1e-3)


def test_camera_rejects_skewed_row():
    K = RO.TEMPLATE_K.copy()
    K[1, 0] = 1.0
    with pytest.raises(ValueError):
        camera.projection_matrix(K, 720, 540, 10.0, 10000.0)


def _quad_verts(z=700.0, half=40.0):
    pts = np.array([[-half, -half, 0], [half, -half, 0], [half, half, 0], [-half, half, 0]], np.float32)
    verts = np.zeros((4, 9), np.float32)
    verts[:, :3] = pts
    verts[:, 5] = -1.0                     # facing the camera (camera looks along +z in OpenCV coordinates)
    verts[:, 6:] = np.float32(0.5)
    return verts, np.array([[0, 1, 2], [0, 2, 3]], np.int32)


def _mats(R=np.eye(3), t=(0.0, 0.0, 700.0), W=720, H=540):
    view, _ = camera.view_matrices(R, np.array(t))
    return view, camera.projection_matrix(RO.TEMPLATE_K, W, H, 10.0, 10000.0), camera.normal_matrix(view)


def test_screen_aligned_quad_covers_exactly_its_pixels_once():
    verts, faces = _quad_verts()
    view, proj, _ = _mats()
    X, Y, zw, cw, _ = RO.project(view, proj, verts[:, :3], 720, 540)
    vis, hits = RO.rasterise(faces, X, Y, zw, 720, 540, count_hits=True)
    assert hits.max() == 1
    covered = (vis & np.uint64(0xffffffff)) != RO.NO_TRI
    assert np.array_equal(covered, hits == 1)
    # expected set: pixel centres inside [Xmin, Xmax) x [Ymin, Ymax) (top-left rule: left and top edges are inclusive)
    xs = np.arange(720) * 256 + 128
    ys = np.arange(540) * 256 + 128
    want = ((ys[:, None] >= Y.min()) & (ys[:, None] < Y.max())) & ((xs[None, :] >= X.min()) & (xs[None, :] < X.max()))
    assert np.array_equal(covered, want)


def test_closed_mesh_has_no_holes_or_double_hits(sphere):
    model = sphere
    verts, faces = mesh_attributes(model)
    view, proj, _ = _mats(R=np.array([[0.36, 0.48, -0.8], [-0.8, 0.6, 0.0], [0.48, 0.64, 0.6]]))
    X, Y, zw, cw, _ = RO.project(view, proj, verts[:, :3], 720, 540)
    _, hits = RO.rasterise(faces, X, Y, zw, 720, 540, count_hits=True)
    # a ray through a pixel centre crosses a closed surface an even number of times: an odd count is a hole or a double hit
    assert np.all(hits % 2 == 0) and (hits == 2).sum() > 1000
    from scipy import ndimage
    filled = ndimage.binary_fill_holes(hits > 0)
    assert np.array_equal(filled, hits > 0)


def test_plane_at_known_depth():
    verts, faces = _quad_verts(half=60.0)
    view, proj, nm = _mats(t=(0.0, 0.0, 850.0))
    bgr, depth, bb, behind = RO.render(verts, faces, view, proj, nm, (400, 400, 400, 0.4, 0.8, 0.3), 720, 540, 10.0)
    assert not behind
    d = depth[depth > 0]
    assert d.size > 1000 and np.all(np.abs(d - 850.0) < 1e-3)
    assert bb is not None and bb[2] > 0


def test_shading_of_one_triangle_matches_the_formula():
    """evaluated by hand in float64 (the fp32 result agrees to a byte): a = 0.4, d = 0.8, s = 0.3, the 4-vector normalisation
    of the normal weights every vertex by 1 / |(n_eye, 1 - t_eye . n_eye)|"""
    verts, faces = _quad_verts()
    verts[:, 3:6] = [0.0, 0.0, -1.0]
    view, proj, nm = _mats()
    light = (400.0, 400.0, 400.0, 0.4, 0.8, 0.3)
    bgr, depth, _, _ = RO.render(verts, faces, view, proj, nm, light, 720, 540, 10.0)
    # pixel at the image centre: eye point P = (x, y, -700) (view = diag(1, 1, -1) . [I | t]); v_view = -P
    r, c = 270, 360
    K = RO.TEMPLATE_K
    X = np.array([(c + 0.5 - K[0, 2]) / K[0, 0] * 700.0, (r + 0.5 - K[1, 2]) / K[1, 1] * 700.0, 700.0])
    P = np.array([X[0], X[1], -X[2]])
    # normal: nm . (0, 0, -1, 1) with t_eye = (0, 0, -700): n_eye = (0, 0, 1), w = 1 - t_eye . n_eye = 701
    n4 = np.array([0.0, 0.0, 1.0, 701.0])
    N = n4[:3] / np.linalg.norm(n4)
    N = N / np.linalg.norm(N)
    L = np.array(light[:3]) - P
    L /= np.linalg.norm(L)
    V = -P / np.linalg.norm(P)
    Rf = -L - 2 * np.dot(N, -L) * N
    val = 0.4 * 0.5 + 0.8 * max(N.dot(L), 0) * 0.5 + 0.3 * max(Rf.dot(V), 0) * 0.5
    assert abs(int(bgr[r, c, 0]) - round(min(val, 1.0) * 255)) <= 1
    assert abs(depth[r, c] - 700.0) < 1e-3


def test_training_draw_order_matches_the_reference_stream():
    """rand(3) for the rotation, random(3) + rand + rand for the light, uniform + uniform for the offsets, per image"""
    from augmentedautoencoder_b200.ae.dataset import Dataset
    ds = Dataset(None, max_rel_offset=0.2)
    np.random.seed(11)
    Rs, lights, offs = ds.training_draws(3)
    np.random.seed(11)
    for i in range(3):
        r = np.random.rand(3)
        q_r1, q_r2 = np.sqrt(1 - r[0]), np.sqrt(r[0])
        assert np.isclose(np.sqrt((1 + np.trace(Rs[i])) / 4.0), abs(np.cos(2 * np.pi * r[2]) * q_r2), atol=1e-9)
        pos = 1000. * np.random.random(3)
        d = 0.8 + 0.1 * (2 * np.random.rand() - 1)
        s = 0.3 + 0.1 * (2 * np.random.rand() - 1)
        assert np.array_equal(lights[i], [pos[0], pos[1], pos[2], 0.4, d, s])
        assert offs[i, 0] == np.random.uniform(-0.2, 0.2) and offs[i, 1] == np.random.uniform(-0.2, 0.2)
        assert np.allclose(Rs[i].dot(Rs[i].T), np.eye(3), atol=1e-12) and q_r1 >= 0


def test_renderer_refuses_what_is_out_of_scope():
    from augmentedautoencoder_b200.ae.dataset import Dataset
    from augmentedautoencoder_b200.meshrenderer.meshrenderer_phong import Renderer
    with pytest.raises(NotImplementedError):
        Renderer(["/nonexistent.ply"], samples=4)
    with pytest.raises(NotImplementedError):
        Dataset(None, model="cad", model_path="/nonexistent.ply").renderer
    ds = Dataset(None, model="reconst", model_path="/nonexistent.ply")   # lazy: constructing never touches the file
    assert ds.has_gpu_renderer


# ------------------------------------------------------------------------------------------------ against the reference's code
# tests/golden/render_golden.npz is written by tests/golden/make_render_golden.py, which runs the reference's load_ply, Camera,
# Renderer.render (OpenGL stubbed, glReadPixels answered by synthetic frames) and Dataset.render_training_images /
# render_embedding_image_batch / get_training_images.

@pytest.fixture(scope="module")
def golden(golden_dir):
    import os
    return dict(np.load(os.path.join(golden_dir, "render_golden.npz")))


def _synthetic_frame(golden_dir, k):
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("make_render_golden", os.path.join(golden_dir, "make_render_golden.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.synthetic_frame(k)


def test_load_ply_matches_the_reference(golden, golden_dir):
    import os
    m = load_ply(os.path.join(golden_dir, "render_mesh.ply"))
    for k in ("pts", "normals", "colors", "faces"):
        assert np.array_equal(m[k], golden["ply_" + k]), k


def test_camera_data_matches_the_reference(golden):
    for pose, want in zip(golden["cam_pose"], golden["cam_data"]):
        R, t, near, far = pose[:9].reshape(3, 3), pose[9:12], pose[12], pose[13]
        got = camera.camera_data(720, 540, RO.TEMPLATE_K, R, t, near, far)
        assert np.allclose(got, want, rtol=1e-6, atol=0), np.abs(got - want).max()
        assert np.array_equal(got, want)


def test_batched_camera_matrices_equal_the_per_view_ones():
    from augmentedautoencoder_b200.ae.dataset import Dataset
    Rs = Dataset(None, min_n_views=162, num_cyclo=12, radius=700).viewsphere_for_embedding
    ts = np.tile([0.0, 0.0, 700.0], (len(Rs), 1))
    ts[::5, 0] = 17.25
    views, _ = camera.view_matrices_batch(Rs, ts)
    nms = camera.normal_matrices(views)
    for i in range(0, len(Rs), 7):
        v, _ = camera.view_matrices(Rs[i], ts[i])
        assert np.array_equal(views[i], v) and np.array_equal(nms[i], camera.normal_matrix(v)), i


def test_training_draw_stream_matches_the_reference(golden):
    """per image: the pose of both render calls (Camera data) and the light uniforms of x (random) and y (fixed); then the
    state of np.random after the loop"""
    from augmentedautoencoder_b200.ae.dataset import Dataset
    n = len(golden["train_x"])
    np.random.seed(1234)
    Rs, lights, offs = Dataset(None, max_rel_offset="0.20").training_draws(n)
    assert np.array_equal(np.random.rand(4), golden["train_after"])
    t = np.array([0, 0, 700.0])
    uni, loc = golden["train_uniforms"], golden["train_uniform_loc"]
    for i in range(n):
        data = camera.camera_data(720, 540, RO.TEMPLATE_K, Rs[i], t, 10.0, 10000.0)
        assert np.array_equal(data, golden["train_scene_data"][2 * i]) and np.array_equal(data, golden["train_scene_data"][2 * i + 1])
        x = {int(loc[k]): uni[k] for k in range(8 * i, 8 * i + 4)}          # location 1 light, 0 ambient, 2 diffuse, 3 specular
        y = {int(loc[k]): uni[k] for k in range(8 * i + 4, 8 * i + 8)}
        got = lights[i].astype(np.float32)
        assert np.array_equal(x[1], got[:3]) and x[0][0] == got[3] and x[2][0] == got[4] and x[3][0] == got[5]
        assert np.array_equal(y[1], np.float32([400, 400, 400])) and (y[0][0], y[2][0], y[3][0]) == (np.float32(0.4), np.float32(0.8), np.float32(0.3))


def test_training_composition_matches_the_reference(golden, golden_dir):
    """the host composition (bbox, offset, crops, mask) fed the reference's synthetic frames and our draws gives the
    reference's train_x / mask_x / train_y bit for bit"""
    from augmentedautoencoder_b200.ae.dataset import Dataset
    n = len(golden["train_x"])
    np.random.seed(1234)
    ds = Dataset(None, max_rel_offset="0.20", pad_factor="1.2")
    _, _, offs = ds.training_draws(n)
    fx = [_synthetic_frame(golden_dir, 2 * i) for i in range(n)]
    fy = [_synthetic_frame(golden_dir, 2 * i + 1) for i in range(n)]
    x, m, y = ds.training_images_from_frames([f[0] for f in fx], [f[1] for f in fx], [f[0] for f in fy], [f[1] for f in fy], offs)
    assert np.array_equal(x, golden["train_x"]) and np.array_equal(m, golden["mask_x"]) and np.array_equal(y, golden["train_y"])


def test_embedding_batch_matches_the_reference(golden, golden_dir):
    from augmentedautoencoder_b200.ae.dataset import Dataset
    frames = iter([_synthetic_frame(golden_dir, 100 + i) for i in range(4)])
    ds = Dataset(None, renderer=lambda R: next(frames), min_n_views=12, num_cyclo=2, radius=700, pad_factor=1.2)
    batch, bbs = ds.render_embedding_image_batch(0, 4)
    assert np.array_equal(batch, golden["emb_batch"]) and np.array_equal(bbs, golden["emb_obj_bbs"])


def test_get_training_images_loads_the_cache_the_reference_names(golden, tmp_path):
    import configparser
    from augmentedautoencoder_b200.ae.dataset import Dataset
    cfg = configparser.ConfigParser()
    cfg.read_string(str(golden["cache_cfg"]))
    np.savez(str(tmp_path / str(golden["cache_name"])), train_x=golden["train_x"], mask_x=golden["mask_x"], train_y=golden["train_y"])
    ds = Dataset(None)
    name = ds.get_training_images(str(tmp_path), cfg)            # loads: nothing is rendered
    assert name.endswith(str(golden["cache_name"]))
    assert np.array_equal(ds.train_x, golden["train_x"]) and np.array_equal(ds.mask_x, golden["mask_x"])
    assert np.array_equal(ds.noof_obj_pixels, np.count_nonzero(golden["mask_x"] == 0, axis=(1, 2)))
