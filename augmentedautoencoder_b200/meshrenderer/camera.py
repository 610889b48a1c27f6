"""Camera matrices of auto_pose/meshrenderer/gl_utils/camera.py (``Camera.realCamera`` with ``setIntrinsic``, lines 81-96 and
144-173, and ``__glOrtho__``): the OpenCV pose [R | t] and intrinsics K become the float32 view and projection matrices the
phong shader multiplies with.  The arithmetic (float64 products rounded to float32 where the reference stores them, the
float32 pseudo-inverse of the world-from-view matrix) is the reference's, so the matrices agree to the last bit with the
same numpy."""
import numpy as np


def gl_ortho(left, right, bottom, top, near, far):
    return np.array([[2. / (right - left), 0., 0., -(right + left) / (right - left)],
                     [0., 2. / (top - bottom), 0., -(top + bottom) / (top - bottom)],
                     [0., 0., -2. / (far - near), -(far + near) / (far - near)],
                     [0., 0., 0., 1.]], dtype=np.float64)


def projection_matrix(K, W, H, near, far):
    """ortho(0, W, H, 0, near, far) . persp(K), rounded to float32; the image origin is the top-left corner"""
    K = np.asarray(K, dtype=np.float64)
    if K.shape != (3, 3):
        raise ValueError("K must be 3x3, got %s" % (K.shape,))
    if K[1, 0] != 0.0 or K[2, 0] != 0.0 or K[2, 1] != 0.0:
        raise ValueError("K[1,0], K[2,0] and K[2,1] must be 0")
    A, B = near + far, near * far
    persp = np.array([[K[0, 0], K[0, 1], -K[0, 2], 0], [0, K[1, 1], -K[1, 2], 0], [0, 0, A, B], [0, 0, -1, 0]], dtype=np.float64)
    return np.dot(gl_ortho(0, W, H, 0, near, far), persp).astype(np.float32)


def view_matrices(R, t):
    """(view = T_view_world, T_world_view), float32: T_world_view = [R^T | -R^T t] . diag(1, 1, -1, 1) and its pseudo-inverse"""
    R = np.asarray(R, dtype=np.float64)[:3, :3]
    t = np.asarray(t, dtype=np.float64)
    world_view = np.eye(4, dtype=np.float32)
    world_view[:3, :3] = R.transpose()
    world_view[:3, 3] = -np.dot(R.transpose(), t.squeeze())
    z_flip = np.eye(4, dtype=np.float32)
    z_flip[2, 2] = -1
    world_view = world_view.dot(z_flip)
    return np.linalg.pinv(world_view), world_view


def view_matrices_batch(Rs, ts):
    """view_matrices for a stack of poses, Rs [n,3,3], ts [n,3]: the same float32 values as the per-view calls (the stacked
    pseudo-inverse runs the same LAPACK routine on every matrix), without a Python loop"""
    Rs = np.asarray(Rs, dtype=np.float64)[:, :3, :3]
    ts = np.asarray(ts, dtype=np.float64).reshape(-1, 3)
    RT = np.transpose(Rs, (0, 2, 1))
    world_view = np.tile(np.eye(4, dtype=np.float32), (len(Rs), 1, 1))
    world_view[:, :3, :3] = RT
    world_view[:, :3, 3] = -np.matmul(RT, ts[:, :, None])[:, :, 0]
    z_flip = np.eye(4, dtype=np.float32)
    z_flip[2, 2] = -1
    world_view = np.matmul(world_view, z_flip)
    return np.linalg.pinv(world_view), world_view


def camera_data(W, H, K, R, t, near, far):
    """The shader storage block of the reference's ``Camera().realCamera(...).data``: view and projection (column-major as
    GLSL reads them) and the camera position, float32 [35]."""
    view, world_view = view_matrices(R, t)
    proj = projection_matrix(K, W, H, near, far)
    return np.hstack((view.T.reshape(-1), proj.T.reshape(-1), world_view[:3, 3].reshape(-1))).astype(np.float32)


def normal_matrix(view):
    """transpose(inverse(view)) of the vertex shader, evaluated in float64 and rounded to float32"""
    return np.linalg.inv(np.asarray(view, dtype=np.float64)).T.astype(np.float32)


def normal_matrices(views):
    """normal_matrix of a stack of view matrices [n,4,4]"""
    return np.transpose(np.linalg.inv(np.asarray(views, dtype=np.float64)), (0, 2, 1)).astype(np.float32)
