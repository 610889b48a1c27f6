"""numpy restatement of the CUDA mesh renderer (augmentedautoencoder_b200/csrc/render.cu), test-only.

What it restates, and from where:
* vertex shader    auto_pose/meshrenderer/shader/depth_shader_phong.vs:20-31 -- P = view . (pos, 1), v_view = -P.xyz,
                   v_L = normalize(light - P.xyz), v_normal = normalize(transpose(inverse(view)) . (n, 1)).xyz (a 4-vector
                   normalisation), v_color;
* fragment shader  shader/depth_shader_phong.frag:20-40 -- ambient + diffuse max(N.L, 0) + specular max(reflect(-L, N).V, 0),
                   no exponent, each channel clamped above at 1; depth = v_view.z;
* fixed function   GL_DEPTH_TEST / GL_LESS on window depth cleared to 1 (meshrenderer_phong.py:92-93,102), GL_RGB8 colour
                   (round(rgb * 255)), glReadPixels(GL_BGR) + flipud (meshrenderer_phong.py:150-157);
* camera           gl_utils/camera.py:81-96,144-173 (augmentedautoencoder_b200/meshrenderer/camera.py builds the matrices).

Every float step is a float32 numpy operation (each one IEEE-rounded, no fused multiply-add) in the order render.cu writes
down; coverage is integer: 8 sub-pixel bits, int64 edge functions, top-left rule, pixel centres.  So the GPU must agree bit
for bit.  Also: seeded test meshes written as .ply (ascii or binary)."""
import numpy as np

F = np.float32
SUB = 256
SNAP = F(536870912.0)
EMPTY = (np.uint64(0x3f800000) << np.uint64(32)) | np.uint64(0xffffffff)
NO_TRI = 0xffffffff


# ------------------------------------------------------------------------------------------------------------ vertex stage
def _row(M, r, x, y, z, w):
    return ((M[r, 0] * x + M[r, 1] * y) + M[r, 2] * z) + M[r, 3] * w


def project(view, proj, pos, W, H):
    """window position of every vertex: X, Y (int64, 8 sub-pixel bits, image rows from the top), window depth zw, clip w,
    camera z (float32)"""
    view, proj = np.asarray(view, F), np.asarray(proj, F)
    x, y, z = pos[:, 0], pos[:, 1], pos[:, 2]
    one = np.ones_like(x)
    P = [_row(view, r, x, y, z, one) for r in range(4)]
    c = [_row(proj, r, P[0], P[1], P[2], P[3]) for r in range(4)]
    halfW, halfH = F(0.5) * F(W), F(0.5) * F(H)
    sx = (c[0] / c[3] + F(1)) * halfW
    sy = (F(1) - c[1] / c[3]) * halfH
    X = np.rint(np.clip(sx * F(SUB), -SNAP, SNAP)).astype(np.int64)
    Y = np.rint(np.clip(sy * F(SUB), -SNAP, SNAP)).astype(np.int64)
    zw = (c[2] / c[3] + F(1)) * F(0.5)
    return X, Y, zw, c[3], -P[2]


def _first_px(lo):
    return -((128 - lo) >> 8)


def _last_px(hi):
    return (hi - 128) >> 8


def _orient(ax, ay, bx, by, cx, cy):
    return (bx - ax) * (cy - ay) - (by - ay) * (cx - ax)


def _bias(ax, ay, bx, by):
    dx, dy = bx - ax, by - ay
    return np.where((dy < 0) | ((dy == 0) & (dx > 0)), 0, -1)


def setup(faces, X, Y):
    """triangles with positive orientation: vertex indices [m, 3] (v1 and v2 swapped where the orientation was negative), A,
    and a validity mask (A != 0)"""
    idx = faces.astype(np.int64).copy()
    A = _orient(X[idx[:, 0]], Y[idx[:, 0]], X[idx[:, 1]], Y[idx[:, 1]], X[idx[:, 2]], Y[idx[:, 2]])
    neg = A < 0
    idx[neg, 1], idx[neg, 2] = faces[neg, 2], faces[neg, 1]
    return idx, np.abs(A), A != 0


def edges(idx, X, Y, px, py):
    cx, cy = px * SUB + SUB // 2, py * SUB + SUB // 2
    x0, y0, x1, y1, x2, y2 = X[idx[:, 0]], Y[idx[:, 0]], X[idx[:, 1]], Y[idx[:, 1]], X[idx[:, 2]], Y[idx[:, 2]]
    return (_orient(x1, y1, x2, y2, cx, cy), _orient(x2, y2, x0, y0, cx, cy), _orient(x0, y0, x1, y1, cx, cy))


def view_box(X, Y, W, H):
    return (max(_first_px(int(X.min())), 0), max(_first_px(int(Y.min())), 0), min(_last_px(int(X.max())), W - 1),
            min(_last_px(int(Y.max())), H - 1))


def rasterise(faces, X, Y, zw, W, H, count_hits=False):
    """visibility keys [H, W] uint64 (depth bits << 32 | triangle); with count_hits also the number of triangles whose
    coverage includes each pixel (before the depth test and the depth range)"""
    vis = np.full(H * W, EMPTY, dtype=np.uint64)
    hits = np.zeros(H * W, np.int64)
    bx0, by0, bx1, by1 = view_box(X, Y, W, H)
    idx, A, ok = setup(faces, X, Y)
    Xs, Ys = X[idx], Y[idx]
    x0 = np.maximum(_first_px(Xs.min(1)), bx0)
    y0 = np.maximum(_first_px(Ys.min(1)), by0)
    x1 = np.minimum(_last_px(Xs.max(1)), bx1)
    y1 = np.minimum(_last_px(Ys.max(1)), by1)
    bw, bh = x1 - x0 + 1, y1 - y0 + 1
    n = np.where(ok & (bw > 0) & (bh > 0), bw * bh, 0)
    tri = np.repeat(np.arange(len(faces)), n)
    local = np.arange(n.sum()) - np.repeat(np.cumsum(n) - n, n)
    px = x0[tri] + local % bw[tri]
    py = y0[tri] + local // bw[tri]
    sub = idx[tri]
    w0, w1, w2 = edges(sub, X, Y, px, py)
    b0 = _bias(X[sub[:, 1]], Y[sub[:, 1]], X[sub[:, 2]], Y[sub[:, 2]])
    b1 = _bias(X[sub[:, 2]], Y[sub[:, 2]], X[sub[:, 0]], Y[sub[:, 0]])
    b2 = _bias(X[sub[:, 0]], Y[sub[:, 0]], X[sub[:, 1]], Y[sub[:, 1]])
    inside = (w0 + b0 >= 0) & (w1 + b1 >= 0) & (w2 + b2 >= 0)
    if count_hits:
        np.add.at(hits, (py * W + px)[inside], 1)
    fA = A[tri].astype(F)
    l0, l1, l2 = w0.astype(F) / fA, w1.astype(F) / fA, w2.astype(F) / fA
    z = (l0 * zw[sub[:, 0]] + l1 * zw[sub[:, 1]]) + l2 * zw[sub[:, 2]]
    keep = inside & (z >= F(0)) & (z < F(1))
    key = (z[keep].view(np.uint32).astype(np.uint64) << np.uint64(32)) | tri[keep].astype(np.uint64)
    np.minimum.at(vis, (py * W + px)[keep], key)
    vis = vis.reshape(H, W)
    return (vis, hits.reshape(H, W)) if count_hits else vis


# ------------------------------------------------------------------------------------------------------------ shading
def _normalize(x, y, z):
    n = np.sqrt((x * x + y * y) + z * z)
    return x / n, y / n, z / n


def _dot(a, b):
    return (a[0] * b[0] + a[1] * b[1]) + a[2] * b[2]


def varyings(verts, view, nm, light):
    """per vertex [12, V]: v_view, v_L, v_normal, v_color (depth_shader_phong.vs)"""
    view, nm = np.asarray(view, F), np.asarray(nm, F)
    light = np.asarray(light, F)
    x, y, z = verts[:, 0], verts[:, 1], verts[:, 2]
    one = np.ones_like(x)
    P = [_row(view, r, x, y, z, one) for r in range(3)]
    L = _normalize(light[0] - P[0], light[1] - P[1], light[2] - P[2])
    n = [_row(nm, r, verts[:, 3], verts[:, 4], verts[:, 5], one) for r in range(4)]
    n4 = np.sqrt(((n[0] * n[0] + n[1] * n[1]) + n[2] * n[2]) + n[3] * n[3])
    return np.stack([-P[0], -P[1], -P[2], L[0], L[1], L[2], n[0] / n4, n[1] / n4, n[2] / n4, verts[:, 6], verts[:, 7], verts[:, 8]])


def shade(verts, faces, X, Y, cw, view, nm, light, px, py, tri):
    """bgr uint8 [k, 3] and depth float32 [k] of the fragments of triangles tri at pixels (px, py)"""
    light = np.asarray(light, F)
    a, d, s = light[3], light[4], light[5]
    idx, A, _ = setup(faces[tri], X, Y)
    w = edges(idx, X, Y, px, py)
    fA = A.astype(F)
    q = [(w[k].astype(F) / fA) / cw[idx[:, k]] for k in range(3)]
    ssum = (q[0] + q[1]) + q[2]
    r = [q[k] / ssum for k in range(3)]
    V = varyings(verts, view, nm, light)
    acc = (r[0] * V[:, idx[:, 0]] + r[1] * V[:, idx[:, 1]]) + r[2] * V[:, idx[:, 2]]
    depth = acc[2]
    Vv = _normalize(acc[0], acc[1], acc[2])
    Lv = _normalize(acc[3], acc[4], acc[5])
    N = _normalize(acc[6], acc[7], acc[8])
    diff = np.fmax(_dot(N, Lv), F(0))
    two_d = F(2) * _dot(N, (-Lv[0], -Lv[1], -Lv[2]))
    R = (-Lv[0] - two_d * N[0], -Lv[1] - two_d * N[1], -Lv[2] - two_d * N[2])
    spec = np.fmax(_dot(R, Vv), F(0))
    bgr = np.empty((len(tri), 3), np.uint8)
    for c in range(3):
        col = acc[9 + c]
        v = np.fmin((a * col + d * (diff * col)) + s * (spec * col), F(1))
        bgr[:, 2 - c] = np.rint(v * F(255)).astype(np.uint8)
    return bgr, depth


def calc_2d_bbox(depth):
    """pysixd_stuff/view_sampler.py:10-15 on depth > 0 (None when nothing was drawn)"""
    ys, xs = np.nonzero(depth > 0)
    if len(xs) == 0:
        return None
    H, W = depth.shape
    x0, y0 = max(xs.min() - 1, 0), max(ys.min() - 1, 0)
    x1, y1 = min(xs.max() + 1, W - 1), min(ys.max() + 1, H - 1)
    return np.array([x0, y0, x1 - x0, y1 - y0], np.int32)


def render(verts, faces, view, proj, nm, light, W, H, near):
    """one full frame: (bgr uint8 [H,W,3], depth float32 [H,W], obj_bb int32 [4] or None, behind-the-camera flag)"""
    X, Y, zw, cw, camz = project(view, proj, verts[:, :3], W, H)
    bgr = np.zeros((H, W, 3), np.uint8)
    depth = np.zeros((H, W), F)
    if not np.all(camz > F(near)):
        return bgr, depth, None, True
    vis = rasterise(faces, X, Y, zw, W, H)
    tri = (vis & np.uint64(0xffffffff)).astype(np.int64)
    py, px = np.nonzero(tri != NO_TRI)
    if len(px):
        c, d = shade(verts, faces, X, Y, cw, view, nm, light, px, py, tri[py, px])
        bgr[py, px] = c
        depth[py, px] = d
    return bgr, depth, calc_2d_bbox(depth), False


# ------------------------------------------------------------------------------------------------------------ test meshes
def _subdivide(verts, faces):
    e = np.sort(np.concatenate([faces[:, [0, 1]], faces[:, [1, 2]], faces[:, [2, 0]]]), axis=1)
    uniq, inv = np.unique(e, axis=0, return_inverse=True)
    mid = len(verts) + inv.reshape(3, -1).T               # [m, 3]: midpoint of edges 01, 12, 20
    verts = np.vstack([verts, 0.5 * (verts[uniq[:, 0]] + verts[uniq[:, 1]])])
    a, b, c = faces.T
    m01, m12, m20 = mid.T
    faces = np.concatenate([np.stack([a, m01, m20], 1), np.stack([m01, b, m12], 1), np.stack([m01, m12, m20], 1),
                            np.stack([m20, m12, c], 1)])
    return verts, faces


def _vertex_normals(pts, faces):
    fn = np.cross(pts[faces[:, 1]] - pts[faces[:, 0]], pts[faces[:, 2]] - pts[faces[:, 0]])
    n = np.zeros_like(pts)
    for k in range(3):
        np.add.at(n, faces[:, k], fn)
    return n / np.linalg.norm(n, axis=1, keepdims=True)


def bumpy_sphere(level, seed=0, radius=60.0, colors=True):
    """closed, asymmetric, outward-oriented sphere with bumps: 20 * 4**level triangles (level 3: 1280, 5: 20480, 6: 81920);
    per-vertex normals and (optionally) colours"""
    from augmentedautoencoder_b200.ae.dataset import _ICO_FACES, _ICO_VERTS
    rng = np.random.RandomState(seed)
    v = np.array(_ICO_VERTS, np.float64)
    f = np.array(_ICO_FACES, np.int64)
    for _ in range(level):
        v, f = _subdivide(v, f)
    u = v / np.linalg.norm(v, axis=1, keepdims=True)
    k = rng.randn(4, 3)
    bump = 0.12 * np.sin(3.0 * u.dot(k[0])) + 0.08 * np.cos(5.0 * u.dot(k[1])) + 0.15 * np.maximum(u.dot(k[2] / np.linalg.norm(k[2])), 0) ** 3
    pts = u * radius * (1.0 + bump)[:, None] * np.array([1.0, 0.8, 1.25])
    # make every face wind outwards (counter-clockwise seen from outside)
    fn = np.cross(pts[f[:, 1]] - pts[f[:, 0]], pts[f[:, 2]] - pts[f[:, 0]])
    flip = np.einsum("ij,ij->i", fn, pts[f].mean(1)) < 0
    f[flip] = f[flip][:, [0, 2, 1]]
    model = {"pts": pts, "normals": _vertex_normals(pts, f), "faces": f}
    if colors:
        model["colors"] = np.clip(np.rint(128 + 100 * np.stack([u.dot(k[3]), u[:, 2], -u[:, 0]], 1)), 0, 255)
    return model


def color_box(size=(150.0, 100.0, 80.0)):
    """axis-aligned box with flat faces (4 vertices each, outward normals, one colour per face): 12 large triangles whose
    shared diagonals and edges exercise the fill rule"""
    sx, sy, sz = np.asarray(size) / 2.0
    pts, nrm, col, faces = [], [], [], []
    palette = [(200, 40, 40), (40, 200, 40), (40, 40, 200), (200, 200, 40), (200, 40, 200), (40, 200, 200)]
    for axis in range(3):
        for sign in (-1.0, 1.0):
            n = np.zeros(3)
            n[axis] = sign
            a, b = [i for i in range(3) if i != axis]
            corners = []
            for ua, ub in ((-1, -1), (1, -1), (1, 1), (-1, 1)):
                p = np.zeros(3)
                p[axis], p[a], p[b] = sign, ua, ub
                corners.append(p * (sx, sy, sz))
            base = len(pts)
            tri = [(0, 1, 2), (0, 2, 3)]
            e = np.cross(corners[1] - corners[0], corners[2] - corners[0])
            if e.dot(n) < 0:
                tri = [(0, 2, 1), (0, 3, 2)]
            pts += corners
            nrm += [n] * 4
            col += [palette[len(faces) // 2]] * 4
            faces += [(base + i, base + j, base + k) for i, j, k in tri]
    return {"pts": np.array(pts), "normals": np.array(nrm), "colors": np.array(col, np.float64), "faces": np.array(faces, np.int64)}


def write_ply(path, model, binary=False):
    """the model as a PLY file with float vertices, uchar colours and int indices"""
    n, m = len(model["pts"]), len(model["faces"])
    has_c = "colors" in model
    head = ["ply", "format %s 1.0" % ("binary_little_endian" if binary else "ascii"), "element vertex %d" % n,
            "property float x", "property float y", "property float z", "property float nx", "property float ny", "property float nz"]
    if has_c:
        head += ["property uchar red", "property uchar green", "property uchar blue"]
    head += ["element face %d" % m, "property list uchar int vertex_indices", "end_header"]
    pts, nrm = model["pts"].astype(np.float32), model["normals"].astype(np.float32)
    with open(path, "wb") as f:
        f.write(("\n".join(head) + "\n").encode())
        if binary:
            fields = [(k, "<f4") for k in ("x", "y", "z", "nx", "ny", "nz")] + ([(k, "u1") for k in ("r", "g", "b")] if has_c else [])
            rec = np.zeros(n, np.dtype(fields))
            for i, k in enumerate(("x", "y", "z")):
                rec[k] = pts[:, i]
            for i, k in enumerate(("nx", "ny", "nz")):
                rec[k] = nrm[:, i]
            if has_c:
                for i, k in enumerate(("r", "g", "b")):
                    rec[k] = model["colors"][:, i].astype(np.uint8)
            f.write(rec.tobytes())
            fr = np.zeros(m, np.dtype([("n", "u1"), ("i", "<i4", (3,))]))
            fr["n"] = 3
            fr["i"] = model["faces"]
            f.write(fr.tobytes())
        else:
            lines = []
            for i in range(n):
                vals = ["%r" % float(v) for v in pts[i]] + ["%r" % float(v) for v in nrm[i]]
                if has_c:
                    vals += ["%d" % int(c) for c in model["colors"][i]]
                lines.append(" ".join(vals))
            lines += ["3 %d %d %d" % tuple(fc) for fc in model["faces"]]
            f.write(("\n".join(lines) + "\n").encode())
    return path


TEMPLATE_K = np.array([[1075.65, 0, 720 / 2], [0, 1073.90, 540 / 2], [0, 0, 1]])
