"""Codebook: cosine nearest-neighbour of the latent against the per-object rotation codebook + 6D pose lift.
Mirrors auto_pose/ae/codebook.py:16-219 (constructor, nearest_rotation, auto_pose6d, nearest_rotation_batch,
test_embedding, update_embedding and the graph attributes callers read).

Differences by design (B200-first): the [B, N] cosine matrix is never copied to the host -- normalise, score and
arg-max/top-k run in one CUDA pass (aae_codebook_match) and only [B, k] (score, index) pairs come back; the matrix is
still available through ``session.run(codebook.cos_similarity, ...)`` for callers that want it.
"""
import ctypes as C

import numpy as np
import torch

from .. import _lib
from . import utils as u
from .session import Placeholder, Tensor, Variable, to_device_input


class Codebook(object):

    def __init__(self, encoder, dataset, embed_bb, precision=None, max_batch=None):
        self._encoder = encoder
        self._dataset = dataset
        self.embed_bb = embed_bb
        self._explicit_precision = precision is not None
        self.precision = encoder.precision if precision is None else int(precision)
        self.max_batch = int(max_batch or encoder.max_batch)

        J = encoder.latent_space_size
        embedding_size = self._dataset.embedding_size
        self._J, self._N = J, embedding_size
        self._handles = {}   # device index -> (handle, version)
        self._version = 0

        self.normalized_embedding_query = Tensor("l2_normalize", (None, J), np.float32, self._eval_zq)
        self.embedding_normalized = Variable(np.zeros((embedding_size, J)), dtype=np.float32, trainable=False,
                                             name="embedding_normalized")
        self.embedding_normalized.on_assign = self._bump
        self.embedding = Placeholder(np.float32, [embedding_size, J], "embedding")
        self.embedding_assign_op = Tensor("assign", (), None, lambda ctx: self.embedding_normalized.assign(ctx.get(self.embedding)))
        if embed_bb:
            self.embed_obj_bbs_var = Variable(np.zeros((embedding_size, 4)), dtype=np.int32, trainable=False, name="embed_obj_bbs_var")
            self.embed_obj_bbs = Placeholder(np.int32, [embedding_size, 4], "embed_obj_bbs")
            self.embed_obj_bbs_assign_op = Tensor("assign_1", (), None, lambda ctx: self.embed_obj_bbs_var.assign(ctx.get(self.embed_obj_bbs)))
            self.embed_obj_bbs_values = None
        self.cos_similarity = Tensor("MatMul", (None, embedding_size), np.float32, self._eval_cos)
        self.nearest_neighbor_idx = Tensor("ArgMax", (None,), np.int64, lambda ctx: self._match(ctx, 1, False)[1][:, 0].to(torch.int64))

    # ------------------------------------------------------------------ device plumbing
    def _bump(self, _value=None):
        self._version += 1

    @property
    def num_cyclo(self):
        return int(self._dataset._kw["num_cyclo"])

    def handle(self, device):
        dev = device.index if isinstance(device, torch.device) else int(device)
        ent = self._handles.get(dev)
        if ent is None or ent[1] != self._version:
            if ent is not None:
                _lib.lib().aae_codebook_destroy(ent[0])
            E = np.ascontiguousarray(self.embedding_normalized.value(), dtype=np.float32)
            h = C.c_void_p()
            with torch.cuda.device(dev):
                self._encoder.handle(dev)                       # settles the encoder's (possibly automatic) precision first
                prec = self.precision if self._explicit_precision else self._encoder.precision
                st = _lib.lib().aae_codebook_create(dev, _lib.ptr(E), E.shape[0], E.shape[1], self.num_cyclo, 0, self.max_batch, prec, C.byref(h))
                if st == -3 and not self._explicit_precision and prec == _lib.PREC_TC_SPLIT:   # e.g. latent != 128: fp32 CUDA-core match
                    prec = _lib.PREC_FP32_SIMT
                    st = _lib.lib().aae_codebook_create(dev, _lib.ptr(E), E.shape[0], E.shape[1], self.num_cyclo, 0, self.max_batch, prec, C.byref(h))
                _lib.check(st, "codebook create")
                self.precision = prec
            self._handles[dev] = (h, self._version)
        return self._handles[dev][0]

    def match_device(self, z_dev, k=1, upright=False):
        """z_dev: CUDA tensor [B, J] (un-normalised latent).  Returns (scores [B,k] float32, idx [B,k] int32) on the device."""
        dev = z_dev.device
        h = self.handle(dev)
        B = z_dev.shape[0]
        scores = torch.empty((B, k), dtype=torch.float32, device=dev)
        idx = torch.empty((B, k), dtype=torch.int32, device=dev)
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        for a in range(0, B, self.max_batch):
            e = min(B, a + self.max_batch)
            _lib.check(_lib.lib().aae_codebook_match(h, _lib.ptr(z_dev[a:e]), e - a, int(k), int(bool(upright)),
                                                     _lib.ptr(scores[a:e]), _lib.ptr(idx[a:e]), stream), "codebook match")
        return scores, idx

    def nearest_idx_device(self, x_dev, k=1, upright=False):
        """crops (CUDA uint8/float32 NHWC) -> (scores, idx) without leaving the device: encoder + fused match."""
        return self.match_device(self._encoder.encode_device(x_dev), k, upright)

    def _match(self, ctx, k, upright):
        return self.match_device(ctx.get(self._encoder.z), k, upright)

    def _eval_zq(self, ctx):
        z = ctx.get(self._encoder.z)
        out = torch.empty_like(z)
        _lib.check(_lib.lib().aae_l2_normalize(_lib.ptr(z), z.shape[0], z.shape[1], _lib.ptr(out), C.c_void_p(ctx.session.stream_ptr)), "l2_normalize")
        return out

    def _eval_cos(self, ctx):
        z = ctx.get(self._encoder.z)
        h = self.handle(z.device)
        B = z.shape[0]
        out = torch.empty((B, self._N), dtype=torch.float32, device=z.device)
        for a in range(0, B, self.max_batch):
            e = min(B, a + self.max_batch)
            _lib.check(_lib.lib().aae_codebook_cosine(h, _lib.ptr(z[a:e]), e - a, _lib.ptr(out[a:e]), C.c_void_p(ctx.session.stream_ptr)), "cosine")
        return out

    # ------------------------------------------------------------------ reference surface
    def nearest_rotation(self, session, x, top_n=1, upright=False, return_idcs=False):
        """R_model2cam of the best codebook row(s) (auto_pose/ae/codebook.py:55-75).  uint8 crops are divided by 255 inside
        the first kernel (a true fp32 divide -- identical to the reference's float64 x/255. rounded at the feed)."""
        if not isinstance(x, torch.Tensor):
            x = np.asarray(x)
        if x.ndim == 3:
            x = x[None]
        xd = to_device_input(x, session.device)
        with torch.cuda.device(session.device):
            _, idx = self.nearest_idx_device(xd, k=top_n, upright=upright)
        idx = idx.cpu().numpy().astype(np.int64)
        self._encoder.check_range(session.device)      # synchronised by the copy above: out-of-range activations raise instead of passing as indices
        if top_n == 1:
            idcs = idx[:, 0]
        else:
            # the reference squeezes the cosine matrix, i.e. top_n > 1 is defined for one crop; keep [B, k] otherwise
            idcs = idx[0] if idx.shape[0] == 1 else idx
        if return_idcs:
            return idcs
        return self._dataset.viewsphere_for_embedding[idcs].squeeze()

    def nearest_rotation_async(self, session, x, upright=False):
        """Non-blocking variant for streaming callers: the host->device copy of `x` (ideally a pinned uint8 tensor) runs on
        the session's copy stream, the encoder + fused match on the compute stream, and the [B] indices come back through a
        pinned buffer.  Returns a ``PendingIndices``; ``.result()`` yields what ``nearest_rotation(..., return_idcs=True)``
        would.  Issue call i+1 before collecting call i to overlap the PCIe copy with the previous batch's compute."""
        dev = session.device
        if not isinstance(x, torch.Tensor):
            a = np.asarray(x)
            x = torch.from_numpy(np.ascontiguousarray(a if a.dtype == np.uint8 else a.astype(np.float32)))
        if x.ndim == 3:
            x = x[None]
        with torch.cuda.device(dev):
            compute = torch.cuda.current_stream(dev)
            copy = session.copy_stream
            with torch.cuda.stream(copy):
                xd = x.to(dev, non_blocking=True)
                if xd.dtype != torch.uint8:
                    xd = xd.to(torch.float32)
                ready = torch.cuda.Event()
                ready.record(copy)
            xd.record_stream(compute)
            compute.wait_event(ready)
            _, idx = self.nearest_idx_device(xd.contiguous(), k=1, upright=upright)
            host = self._pinned_result(idx.shape)
            host.copy_(idx, non_blocking=True)
            # the range guard's word rides behind the indices on the same stream: no extra synchronisation in the pipeline
            word = self._encoder.range_word(dev)
            flag = None
            if word is not None:
                flag = self._pinned_result((1,))
                flag.copy_(word, non_blocking=True)
            done = torch.cuda.Event()
            done.record(compute)
        return PendingIndices(host, done, flag, lambda: self._encoder.check_range(dev))

    def _pinned_result(self, shape, depth=8):
        """Ring of pinned host buffers for the async read-back (cudaHostAlloc per call would cost more than the kernel)."""
        ring = self.__dict__.setdefault("_pin_ring", {})
        key = tuple(shape)
        bufs, pos = ring.get(key, ([], 0))
        if len(bufs) < depth:
            bufs.append(torch.empty(key, dtype=torch.int32, pin_memory=True))
            buf = bufs[-1]
        else:
            buf = bufs[pos % depth]
        ring[key] = (bufs, pos + 1)
        return buf

    def auto_pose6d(self, session, x, predicted_bb, K_test, top_n, train_args, depth_pred=None, upright=False):
        """Rotation from the codebook + translation from the bbox-diagonal ratio + rotation correction
        (auto_pose/ae/codebook.py:79-129)."""
        idcs = np.atleast_1d(self.nearest_rotation(session, x, top_n=top_n, upright=upright, return_idcs=True))
        K_train = np.array(eval(train_args.get("Dataset", "K"))).reshape(3, 3)
        render_radius = train_args.getfloat("Dataset", "RADIUS")
        if self.embed_obj_bbs_values is None:
            self.embed_obj_bbs_values = session.run(self.embed_obj_bbs_var)
        return lift_pose(idcs, self._dataset.viewsphere_for_embedding, self.embed_obj_bbs_values, predicted_bb,
                         np.asarray(K_test), K_train, render_radius, depth_pred)

    def nearest_rotation_batch(self, session, x):
        idcs = session.run(self.nearest_neighbor_idx, {self._encoder.x: x})
        return self._dataset.viewsphere_for_embedding[idcs]

    def test_embedding(self, sess, x, normalized=True):
        if not isinstance(x, torch.Tensor):
            x = np.asarray(x)
        if x.ndim == 3:
            x = x[None]
        fetch = self.normalized_embedding_query if normalized else self._encoder.z
        return sess.run(fetch, {self._encoder.x: x}).squeeze()

    def update_embedding(self, session, batch_size):
        """Build the codebook: encode every rendered view, L2-normalise in float64, store fp32 (codebook.py:190-219).  With the
        dataset's CUDA renderer the uint8 crops go from the renderer to the encoder without a host round trip."""
        if getattr(self._dataset, "has_gpu_renderer", False):
            return self._update_embedding(session, batch_size, self._dataset.embedding_crops_device)
        return self._update_embedding(session, batch_size, self._dataset.render_embedding_image_batch)

    def update_embedding_from_crops(self, session, crops, obj_bbs=None, batch_size=256):
        """Same as update_embedding for pre-rendered view crops ([N,H,W,C] uint8 or float in [0,1])."""
        if len(crops) != self._N:
            raise ValueError("need %d crops (one per view-sphere rotation), got %d" % (self._N, len(crops)))
        return self._update_embedding(session, batch_size, lambda a, e: (crops[a:e], None if obj_bbs is None else obj_bbs[a:e]))

    def _update_embedding(self, session, batch_size, batch_fn):
        embedding_z = np.empty((self._N, self._J))
        obj_bbs = np.zeros((self._N, 4))
        for a, e in u.batch_iteration_indices(self._N, batch_size):
            batch, bbs = batch_fn(a, e)
            embedding_z[a:e] = session.run(self._encoder.z, feed_dict={self._encoder.x: batch})
            if self.embed_bb and bbs is not None:
                obj_bbs[a:e] = bbs.cpu().numpy() if isinstance(bbs, torch.Tensor) else bbs
        normalized_embedding = embedding_z / np.linalg.norm(embedding_z, axis=1, keepdims=True)
        session.run(self.embedding_assign_op, {self.embedding: normalized_embedding})
        if self.embed_bb:
            session.run(self.embed_obj_bbs_assign_op, {self.embed_obj_bbs: obj_bbs})
            self.embed_obj_bbs_values = None

    def close(self):
        for h, _ in self._handles.values():
            _lib.lib().aae_codebook_destroy(h)
        self._handles = {}

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PendingIndices:
    """Handle returned by Codebook.nearest_rotation_async."""

    def __init__(self, host_buf, event, flag=None, check=None):
        self._host, self._event, self._flag, self._check = host_buf, event, flag, check

    def done(self):
        return self._event.query()

    def result(self):
        self._event.synchronize()
        if self._flag is not None and int(self._flag[0]) != 0:
            self._check()              # synchronises, clears the guard and raises AaeError naming the layers
        return self._host.numpy().astype(np.int64)[:, 0]   # astype copies: the pinned buffer goes back to the ring


def _sq_scalar(a):
    """x**2 exactly as the reference evaluates it: on numpy float64 SCALARS (``t_est[2]**2``, codebook.py:121), which goes
    through C pow() and is not always bit-identical to the array fast path x*x."""
    flat = np.asarray(a, dtype=np.float64).ravel()
    return np.array([v ** 2 for v in flat], dtype=np.float64).reshape(np.shape(a))


def lift_pose_batch(idcs, rs_table, embed_obj_bbs, predicted_bbs, K_test, K_train, render_radius, depth_pred=None):
    """``auto_pose6d``'s numpy tail (auto_pose/ae/codebook.py:82-129) for ALL detections of one object class at once:
    idcs [D, k] codebook rows (k hypotheses per detection), predicted_bbs [D, 4] xywh -> (Rs [D, k, 3, 3], ts [D, k, 3]),
    float64, bit-identical to calling the reference per detection (same operations on the same dtypes in the same order;
    tests/test_host_logic.py checks it against the reference-generated golden and against the per-detection loop)."""
    idcs = np.asarray(idcs)
    if idcs.ndim == 1:
        idcs = idcs[:, None]
    D, k = idcs.shape
    pb = np.asarray(predicted_bbs).reshape(D, 4)
    R = rs_table[idcs]                                           # [D, k, 3, 3]
    rb = np.asarray(embed_obj_bbs)[idcs]                         # [D, k, 4] rendered bounding boxes
    K_diag_ratio = np.sqrt(K_test[0, 0] ** 2 + K_test[1, 1] ** 2) / np.sqrt(K_train[0, 0] ** 2 + K_train[1, 1] ** 2)
    if depth_pred is None:
        r32, p32 = np.float32(rb[..., 2:]), np.float32(pb[:, 2:])
        # np.linalg.norm of a 2-vector of float32 = sqrt(x . x) evaluated in float32
        n_r = np.sqrt(r32[..., 0] * r32[..., 0] + r32[..., 1] * r32[..., 1])
        n_p = np.sqrt(p32[:, 0] * p32[:, 0] + p32[:, 1] * p32[:, 1])
        z = (n_r / n_p[:, None]) * K_diag_ratio * render_radius
    else:
        z = np.broadcast_to(np.asarray(depth_pred, dtype=np.float64).reshape(-1, 1), (D, k)).copy()
    cx_train = rb[..., 0] + rb[..., 2] / 2. - K_train[0, 2]
    cy_train = rb[..., 1] + rb[..., 3] / 2. - K_train[1, 2]
    cx_test = (pb[:, 0] + pb[:, 2] / 2 - K_test[0, 2])[:, None]
    cy_test = (pb[:, 1] + pb[:, 3] / 2 - K_test[1, 2])[:, None]
    tx = cx_test * z / K_test[0, 0] - cx_train * render_radius / K_train[0, 0]
    ty = cy_test * z / K_test[1, 1] - cy_train * render_radius / K_train[1, 1]
    z = z.astype(np.float64)
    ts = np.stack([tx, ty, z], axis=-1).astype(np.float64)
    ay = np.arctan(ts[..., 0] / np.sqrt(_sq_scalar(ts[..., 2]) + _sq_scalar(ts[..., 1])))
    ax = -np.arctan(ts[..., 1] / ts[..., 2])
    cax, sax, cay, say = np.cos(ax), np.sin(ax), np.cos(ay), np.sin(ay)
    Rx = np.zeros((D, k, 3, 3))
    Rx[..., 0, 0], Rx[..., 1, 1], Rx[..., 1, 2], Rx[..., 2, 1], Rx[..., 2, 2] = 1, cax, -sax, sax, cax
    Ry = np.zeros((D, k, 3, 3))
    Ry[..., 0, 0], Ry[..., 0, 2], Ry[..., 1, 1], Ry[..., 2, 0], Ry[..., 2, 2] = cay, say, 1, -say, cay
    return np.matmul(Ry, np.matmul(Rx, R)), ts


def lift_pose(idcs, rs_table, embed_obj_bbs, predicted_bb, K_test, K_train, render_radius, depth_pred=None):
    """The numpy tail of Codebook.auto_pose6d (codebook.py:82-129): depth from the ratio of rendered to detected bbox
    diagonals scaled by the focal-length ratio, lateral offset from the bbox centres, and the rotation that keeps the
    appearance when the object is moved off the optical axis."""
    Rs_est = rs_table[idcs].copy()
    K_diag_ratio = np.sqrt(K_test[0, 0] ** 2 + K_test[1, 1] ** 2) / np.sqrt(K_train[0, 0] ** 2 + K_train[1, 1] ** 2)
    ts_est = np.empty((len(idcs), 3))
    for i, idx in enumerate(idcs):
        rendered_bb = embed_obj_bbs[idx].squeeze()
        if depth_pred is None:
            bb_diag_ratio = np.linalg.norm(np.float32(rendered_bb[2:])) / np.linalg.norm(np.float32(predicted_bb[2:]))
            z = bb_diag_ratio * K_diag_ratio * render_radius
        else:
            z = depth_pred
        cx_train = rendered_bb[0] + rendered_bb[2] / 2. - K_train[0, 2]
        cy_train = rendered_bb[1] + rendered_bb[3] / 2. - K_train[1, 2]
        cx_test = predicted_bb[0] + predicted_bb[2] / 2 - K_test[0, 2]
        cy_test = predicted_bb[1] + predicted_bb[3] / 2 - K_test[1, 2]
        tx = cx_test * z / K_test[0, 0] - cx_train * render_radius / K_train[0, 0]
        ty = cy_test * z / K_test[1, 1] - cy_train * render_radius / K_train[1, 1]
        t_est = np.array([tx, ty, z])
        ts_est[i] = t_est
        ay = np.arctan(t_est[0] / np.sqrt(t_est[2] ** 2 + t_est[1] ** 2))
        ax = -np.arctan(t_est[1] / t_est[2])
        R_corr_x = np.array([[1, 0, 0], [0, np.cos(ax), -np.sin(ax)], [0, np.sin(ax), np.cos(ax)]])
        R_corr_y = np.array([[np.cos(ay), 0, np.sin(ay)], [0, 1, 0], [-np.sin(ay), 0, np.cos(ay)]])
        Rs_est[i] = np.dot(R_corr_y, np.dot(R_corr_x, Rs_est[i]))
    return (Rs_est, ts_est)
