"""GPU tests of the CUDA mesh renderer (csrc/render.cu): full frames bit-identical to the numpy restatement
(oracle/render_oracle.py), fused crops bit-identical to Dataset.extract_square_patch (cv2 INTER_NEAREST) of the GPU's own frames,
the device codebook build, the training set, determinism, batch independence and the behind-the-camera guard."""
import numpy as np
import pytest
import torch

from oracle import render_oracle as RO

pytestmark = pytest.mark.gpu

W, H = 720, 540
NEAR, FAR = 10.0, 10000.0
T = np.array([0.0, 0.0, 700.0])


@pytest.fixture(scope="module")
def plys(tmp_path_factory):
    d = tmp_path_factory.mktemp("meshes")
    return {"sphere": RO.write_ply(str(d / "sphere.ply"), RO.bumpy_sphere(3, seed=2)),
            "box": RO.write_ply(str(d / "box.ply"), RO.color_box(), binary=True),
            "plain": RO.write_ply(str(d / "plain.ply"), RO.bumpy_sphere(2, seed=5, colors=False)),
            "big": RO.write_ply(str(d / "big.ply"), RO.bumpy_sphere(6, seed=3), binary=True)}


@pytest.fixture(scope="module")
def renderer(plys):
    from augmentedautoencoder_b200.meshrenderer.meshrenderer_phong import Renderer
    torch.cuda.set_device(0)
    r = Renderer([plys["sphere"], plys["box"], plys["plain"], plys["big"]])
    yield r
    r.close()


def _rotations(n, seed):
    from augmentedautoencoder_b200.ae.dataset import Dataset, random_rotation_matrix
    ds = Dataset(None, min_n_views=42, num_cyclo=4, radius=700)
    np.random.seed(seed)
    rand = [random_rotation_matrix()[:3, :3] for _ in range(n - n // 2)]
    return np.concatenate([ds.viewsphere_for_embedding[::7][:n // 2], np.array(rand)])


@pytest.mark.parametrize("obj_id", [0, 1, 2])
def test_full_frames_match_the_oracle_bit_for_bit(renderer, obj_id, plys):
    from augmentedautoencoder_b200.meshrenderer import camera
    from augmentedautoencoder_b200.meshrenderer.inout import load_ply, mesh_attributes
    from augmentedautoencoder_b200.meshrenderer.meshrenderer_phong import fixed_light, random_light
    Rs = _rotations(16, seed=obj_id)
    np.random.seed(100 + obj_id)
    lights = np.array([fixed_light() if i % 2 == 0 else random_light() for i in range(len(Rs))])
    bgr, depth, bb, flags = renderer.render_frames_device(obj_id, W, H, RO.TEMPLATE_K, Rs, T, NEAR, FAR, lights)
    bgr, depth, bb = bgr.cpu().numpy(), depth.cpu().numpy(), bb.cpu().numpy()
    verts, faces = mesh_attributes(load_ply([plys["sphere"], plys["box"], plys["plain"]][obj_id]))
    proj = camera.projection_matrix(RO.TEMPLATE_K, W, H, NEAR, FAR)
    for i, R in enumerate(Rs):
        view, _ = camera.view_matrices(R, T)
        want_bgr, want_depth, want_bb, behind = RO.render(verts, faces, view, proj, camera.normal_matrix(view),
                                                          lights[i].astype(np.float32), W, H, NEAR)
        assert not behind
        assert np.array_equal(bgr[i], want_bgr), (i, np.argwhere(np.any(bgr[i] != want_bgr, -1))[:5])
        assert np.array_equal(depth[i].view(np.uint32), want_depth.view(np.uint32)), i
        assert np.array_equal(bb[i], want_bb), (i, bb[i], want_bb)
    assert int(flags.abs().sum()) == 0


def _host_crops(ds, bgr, depth, bbs, offsets, pad, size):
    import cv2
    xs, ms = [], []
    for i in range(len(bgr)):
        box = bbs[i].astype(np.float64) + (np.array([offsets[i, 0] * bbs[i, 2], offsets[i, 1] * bbs[i, 3], 0, 0]) if offsets is not None else 0)
        xs.append(ds.extract_square_patch(bgr[i], box, pad, resize=(size, size), interpolation=cv2.INTER_NEAREST))
        ms.append(ds.extract_square_patch(depth[i], box, pad, resize=(size, size), interpolation=cv2.INTER_NEAREST) == 0.)
    return np.array(xs), np.array(ms)


@pytest.mark.parametrize("obj_id", [0, 1, 3])
def test_fused_crops_match_host_crops_of_the_gpu_frames(renderer, obj_id):
    from augmentedautoencoder_b200.ae.dataset import Dataset
    from augmentedautoencoder_b200.meshrenderer.meshrenderer_phong import fixed_light, random_light
    ds = Dataset(None)
    Rs = _rotations(24, seed=10 + obj_id)
    np.random.seed(7)
    lx = np.array([random_light() for _ in Rs])
    offs = np.random.uniform(-0.2, 0.2, (len(Rs), 2))
    offs[:4] = [[-1.6, 0.1], [1.6, -1.5], [0.4, 1.5], [-1.7, -1.4]]    # crop windows clipped at the frame edge
    bgr, depth, bb, _ = renderer.render_frames_device(obj_id, W, H, RO.TEMPLATE_K, Rs, T, NEAR, FAR, lx)
    bgr_y, _, _, _ = renderer.render_frames_device(obj_id, W, H, RO.TEMPLATE_K, Rs, T, NEAR, FAR, fixed_light())
    bgr, depth, bb, bgr_y = bgr.cpu().numpy(), depth.cpu().numpy(), bb.cpu().numpy(), bgr_y.cpu().numpy()
    out = renderer.render_crops_device(obj_id, W, H, RO.TEMPLATE_K, Rs, T, NEAR, FAR, lx, 1.2, 128, 128, lights_y=fixed_light(),
                                       offsets=offs, want_mask=True)
    want_x, want_m = _host_crops(ds, bgr, depth, bb, offs, 1.2, 128)
    want_y, _ = _host_crops(ds, bgr_y, depth, bb, None, 1.2, 128)
    assert np.array_equal(out["obj_bb"].cpu().numpy(), bb)
    assert np.array_equal(out["x"].cpu().numpy(), want_x)
    assert np.array_equal(out["mask"].cpu().numpy(), want_m)
    assert np.array_equal(out["y"].cpu().numpy(), want_y)
    # embedding crops: fixed light, no offsets, no mask
    emb = renderer.render_crops_device(obj_id, W, H, RO.TEMPLATE_K, Rs, T, NEAR, FAR, fixed_light(), 1.2, 128, 128)
    assert np.array_equal(emb["x"].cpu().numpy(), want_y)


def test_determinism_and_batch_independence(renderer):
    from augmentedautoencoder_b200.meshrenderer.meshrenderer_phong import fixed_light
    Rs = _rotations(300, seed=3)
    ref = renderer.render_crops_device(0, W, H, RO.TEMPLATE_K, Rs, T, NEAR, FAR, fixed_light(), 1.2, 128, 128)["x"].cpu().numpy()
    again = renderer.render_crops_device(0, W, H, RO.TEMPLATE_K, Rs, T, NEAR, FAR, fixed_light(), 1.2, 128, 128)["x"].cpu().numpy()
    assert np.array_equal(ref, again)
    for step in (1, 7, 256):
        parts = [renderer.render_crops_device(0, W, H, RO.TEMPLATE_K, Rs[a:a + step], T, NEAR, FAR, fixed_light(), 1.2, 128, 128)["x"]
                 for a in range(0, 40 if step == 1 else len(Rs), step)]
        got = torch.cat(parts).cpu().numpy()
        assert np.array_equal(got, ref[:len(got)]), step
    f1 = renderer.render_frames_device(1, W, H, RO.TEMPLATE_K, Rs[:9], T, NEAR, FAR, fixed_light())[0]
    f2 = torch.cat([renderer.render_frames_device(1, W, H, RO.TEMPLATE_K, Rs[a:min(a + 4, 9)], T, NEAR, FAR, fixed_light())[0]
                    for a in (0, 4, 8)])
    assert torch.equal(f1, f2)


def test_a_vertex_behind_the_camera_names_the_view(renderer):
    from augmentedautoencoder_b200.meshrenderer.meshrenderer_phong import RenderError, fixed_light
    Rs = _rotations(5, seed=4)
    ts = np.tile(T, (5, 1))
    ts[2, 2] = 40.0                                   # the sphere (radius ~75 mm) reaches behind the near plane
    bgr, depth, bb, flags = renderer.render_frames_device(0, W, H, RO.TEMPLATE_K, Rs, ts, NEAR, FAR, fixed_light(), check=False)
    assert (flags.cpu().numpy() & 1).tolist() == [0, 0, 1, 0, 0]
    ok = renderer.render_frames_device(0, W, H, RO.TEMPLATE_K, Rs[[0, 1, 3, 4]], T, NEAR, FAR, fixed_light())[0]
    assert torch.equal(bgr[[0, 1, 3, 4]], ok)
    with pytest.raises(RenderError, match=r"view\(s\) \[2\]"):
        renderer.render_crops_device(0, W, H, RO.TEMPLATE_K, Rs, ts, NEAR, FAR, fixed_light(), 1.2, 128, 128)


def test_obj_id_selects_the_mesh_and_render_matches_the_batch(renderer):
    from augmentedautoencoder_b200.meshrenderer.meshrenderer_phong import fixed_light
    R = _rotations(2, seed=5)[1]
    a, da = renderer.render(0, W, H, RO.TEMPLATE_K, R, T, NEAR, FAR)
    b, db = renderer.render(1, W, H, RO.TEMPLATE_K, R, T, NEAR, FAR)
    assert a.shape == (H, W, 3) and da.dtype == np.float32 and not np.array_equal(a, b)
    box_bgr = renderer.render_frames_device(1, W, H, RO.TEMPLATE_K, [R], T, NEAR, FAR, fixed_light())[0][0].cpu().numpy()
    assert np.array_equal(b, box_bgr)
    np.random.seed(3)
    renderer.render(0, W, H, RO.TEMPLATE_K, R, T, NEAR, FAR, random_light=True)
    np.random.seed(3)
    np.random.random(3), np.random.rand(), np.random.rand()
    after = np.random.rand()
    np.random.seed(3)
    renderer.render(0, W, H, RO.TEMPLATE_K, R, T, NEAR, FAR, random_light=True)
    assert np.random.rand() == after                # random_light consumes random(3), rand, rand


def _dataset(plys, **kw):
    from augmentedautoencoder_b200.ae.dataset import Dataset
    args = dict(model="reconst", model_path=plys["sphere"], antialiasing="1", vertex_scale="1", render_dims="(720, 540)",
                k="[1075.65, 0, 720/2, 0, 1073.90, 540/2, 0, 0, 1]", clip_near="10", clip_far="10000", pad_factor="1.2", radius="700",
                max_rel_offset="0.20", h="128", w="128", c="3")
    args.update(kw)
    return Dataset(None, **args)


def test_device_update_embedding_equals_host_crops(plys):
    from augmentedautoencoder_b200.ae.codebook import Codebook
    from augmentedautoencoder_b200.ae.encoder import Encoder
    from augmentedautoencoder_b200.ae.session import Session, placeholder
    from oracle import aae_oracle as O
    import cv2
    sess = Session(device=0)
    ds = _dataset(plys, min_n_views=42, num_cyclo=8)
    enc = Encoder(placeholder(np.float32, [None, 128, 128, 3]), 128, list(O.NUM_FILTER), 5, list(O.STRIDES), False, precision=0, max_batch=64)
    enc.load_weights(O.make_encoder_params(42, bias_scale=0.05))
    cb = Codebook(enc, ds, True, max_batch=64)
    cb.update_embedding(sess, 64)
    E, bbs = sess.run(cb.embedding_normalized), sess.run(cb.embed_obj_bbs_var)
    # host composition: full frames from Renderer.render, calc_2d_bbox, Dataset.extract_square_patch
    crops, host_bbs = [], []
    for R in ds.viewsphere_for_embedding:
        bgr, depth = ds.renderer.render(0, 720, 540, RO.TEMPLATE_K, R, np.array([0, 0, 700.0]), 10.0, 10000.0)
        bb = RO.calc_2d_bbox(depth)
        host_bbs.append(bb)
        crops.append(ds.extract_square_patch(bgr, bb, 1.2, resize=(128, 128), interpolation=cv2.INTER_NEAREST))
    cb2 = Codebook(enc, ds, True, max_batch=64)
    cb2.update_embedding_from_crops(sess, np.array(crops), np.array(host_bbs), batch_size=64)
    assert np.array_equal(E, sess.run(cb2.embedding_normalized))
    assert np.array_equal(bbs, np.array(host_bbs))
    idc = cb.nearest_rotation(sess, np.array(crops), return_idcs=True)
    # every view finds itself; the first and last in-plane steps of linspace(0, 2 pi, num_cyclo) are the same rotation
    Rv = ds.viewsphere_for_embedding
    assert np.allclose(Rv[idc], Rv, atol=1e-9) and np.mean(idc == np.arange(len(crops))) >= 7 / 8
    batch, obj_bbs = ds.render_embedding_image_batch(0, 5)
    assert np.array_equal(batch, np.array(crops[:5]) / 255.) and np.array_equal(obj_bbs, np.array(host_bbs[:5]))


def test_render_training_images_equals_the_host_composition(plys):
    import cv2
    from augmentedautoencoder_b200.meshrenderer.meshrenderer_phong import random_light
    from augmentedautoencoder_b200.ae.dataset import random_rotation_matrix
    ds = _dataset(plys, noof_training_imgs="64")
    np.random.seed(2024)
    ds.render_training_images()
    state_after = np.random.rand()
    # the reference's loop (dataset.py:238-303) with Renderer.render
    np.random.seed(2024)
    K, t = RO.TEMPLATE_K, np.array([0, 0, 700.0])
    for i in range(64):
        R = random_rotation_matrix()[:3, :3]
        bgr_x, depth_x = ds.renderer.render(0, 720, 540, K, R, t, 10.0, 10000.0, random_light=True)
        bgr_y, depth_y = ds.renderer.render(0, 720, 540, K, R, t, 10.0, 10000.0, random_light=False)
        bb = RO.calc_2d_bbox(depth_x)
        x, y, w, h = bb
        off = bb + np.array([np.random.uniform(-0.2, 0.2) * w, np.random.uniform(-0.2, 0.2) * h, 0, 0])
        cx = ds.extract_square_patch(bgr_x, off, 1.2, resize=(128, 128), interpolation=cv2.INTER_NEAREST)
        cd = ds.extract_square_patch(depth_x, off, 1.2, resize=(128, 128), interpolation=cv2.INTER_NEAREST)
        cy = ds.extract_square_patch(bgr_y, RO.calc_2d_bbox(depth_y), 1.2, resize=(128, 128), interpolation=cv2.INTER_NEAREST)
        assert np.array_equal(ds.train_x[i], cx), i
        assert np.array_equal(ds.mask_x[i], cd == 0.), i
        assert np.array_equal(ds.train_y[i], cy), i
    assert np.random.rand() == state_after
    assert ds.train_x.dtype == np.uint8 and ds.mask_x.dtype == bool and ds.train_y.dtype == np.uint8


@pytest.mark.parametrize("n", [1, 3])
def test_odd_frame_size_and_odd_batch_match_the_oracle(renderer, plys, n):
    """641 x 481 with an odd number of views: every workspace section must stay aligned (W * H * n odd)"""
    from augmentedautoencoder_b200.meshrenderer import camera
    from augmentedautoencoder_b200.meshrenderer.inout import load_ply, mesh_attributes
    from augmentedautoencoder_b200.meshrenderer.meshrenderer_phong import fixed_light
    Wo, Ho = 641, 481
    K = np.array([[1075.65, 0, Wo / 2], [0, 1073.90, Ho / 2], [0, 0, 1]])
    Rs = _rotations(n + 1, seed=20 + n)[:n]
    bgr, depth, bb, _ = renderer.render_frames_device(1, Wo, Ho, K, Rs, T, NEAR, FAR, fixed_light())
    verts, faces = mesh_attributes(load_ply(plys["box"]))
    proj = camera.projection_matrix(K, Wo, Ho, NEAR, FAR)
    for i, R in enumerate(Rs):
        view, _ = camera.view_matrices(R, T)
        wb, wd, wbb, _ = RO.render(verts, faces, view, proj, camera.normal_matrix(view), fixed_light().astype(np.float32), Wo, Ho, NEAR)
        assert np.array_equal(bgr[i].cpu().numpy(), wb) and np.array_equal(depth[i].cpu().numpy().view(np.uint32), wd.view(np.uint32))
        assert np.array_equal(bb[i].cpu().numpy(), wbb)
    out = renderer.render_crops_device(1, Wo, Ho, K, Rs, T, NEAR, FAR, fixed_light(), 1.2, 128, 128)
    from augmentedautoencoder_b200.ae.dataset import Dataset
    want, _ = _host_crops(Dataset(None), bgr.cpu().numpy(), depth.cpu().numpy(), bb.cpu().numpy(), None, 1.2, 128)
    assert np.array_equal(out["x"].cpu().numpy(), want)
