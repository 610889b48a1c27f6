"""Times the CUDA mesh renderer on the GPU: the fused 92 232-view codebook build (render + crop, then encode; the two phases timed
separately with CUDA events) on a 20 k and an 80 k triangle mesh, 20 000 training pairs (x crop + mask + y crop), and, for
comparison, the full-frame path followed by the same crops taken from the frames.  The host setup of the per-view matrices
is timed on its own.  Prints the
card name and power limit first.

    python scripts/time_render.py [--views 92232] [--train 20000] [--out profiles/render_timings.txt]
"""
import argparse
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else torch.cuda.get_device_name(0)


def timed(fn, reps=1):
    fn()                                   # warm-up of every shape
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--views", type=int, default=92232)
    ap.add_argument("--train", type=int, default=20000)
    ap.add_argument("--chunk", type=int, default=4096)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_render.py measures the GPU renderer and needs a CUDA device")
    from augmentedautoencoder_b200 import build_ext
    build_ext.build()
    from augmentedautoencoder_b200.ae.dataset import Dataset
    from augmentedautoencoder_b200.ae.encoder import Encoder
    from augmentedautoencoder_b200.ae.session import placeholder
    from augmentedautoencoder_b200.meshrenderer.meshrenderer_phong import Renderer, fixed_light
    from oracle import aae_oracle as O
    from oracle import render_oracle as RO

    lines = ["card: " + card() + "  (name, power limit, max SM clock)"]
    K, t = RO.TEMPLATE_K, np.array([0, 0, 700.0])
    ds = Dataset(None, min_n_views=2562, num_cyclo=36, radius=700)
    Rs = ds.viewsphere_for_embedding[:args.views]
    enc = Encoder(placeholder(np.float32, [None, 128, 128, 3]), 128, list(O.NUM_FILTER), 5, list(O.STRIDES), False, precision=1,
                  max_batch=args.chunk)
    enc.load_weights(O.make_encoder_params(42, bias_scale=0.05))
    tmp = tempfile.mkdtemp()
    for level, label in ((5, "20k"), (6, "80k")):
        path = RO.write_ply(os.path.join(tmp, "s%d.ply" % level), RO.bumpy_sphere(level, seed=3), binary=True)
        r = Renderer([path])
        lines.append("mesh %s: %d vertices, %d triangles" % (label, r.n_vertices[0], 20 * 4 ** level))

        def crops(a, e):
            return r.render_crops_device(0, 720, 540, K, Rs[a:e], t, 10.0, 10000.0, fixed_light(), 1.2, 128, 128, check=False)["x"]

        # render + crop of all views (chunks of args.chunk views), then the encoder on the same crops, phases timed apart
        chunks = [(a, min(len(Rs), a + args.chunk)) for a in range(0, len(Rs), args.chunk)]
        crops(*chunks[0])
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        render_ms = encode_ms = 0.0
        for a, e in chunks:
            ev[0].record()
            x = crops(a, e)
            ev[1].record()
            enc.encode_device(x)
            ev[2].record()
            torch.cuda.synchronize()
            render_ms += ev[0].elapsed_time(ev[1])
            encode_ms += ev[1].elapsed_time(ev[2])
        n = len(Rs)
        t0 = time.perf_counter()
        for a, e in chunks:
            Renderer._params(720, 540, K, Rs[a:e], t, 10.0, 10000.0, fixed_light())
        host_ms = (time.perf_counter() - t0) * 1e3
        lines.append("  host setup of the per-view matrices (inside the render+crop window below): %.1f ms" % host_ms)
        lines.append("  fused embedding, %d views: render+crop %.1f ms (%.0f views/s), encode %.1f ms (%.0f crops/s)"
                     % (n, render_ms, n / render_ms * 1e3, encode_ms, n / encode_ms * 1e3))
        # full-frame path + the same crops taken from the frames, on the first 2048 views
        m = min(n, 2048)
        sub = Rs[:m]

        cols, rows = (m_.cpu().numpy() for m_ in r._nearest_maps(720, 540, 128, 128))
        vi = torch.arange(m, device=r.device)[:, None, None]

        def frames_then_crop():
            # full frames, then Dataset.extract_square_patch + INTER_NEAREST of every frame: windows on the host from the
            # read-back boxes, one gather on the device
            bgr, depth, bb, _ = r.render_frames_device(0, 720, 540, K, sub, t, 10.0, 10000.0, fixed_light(), check=False)
            x, y, w, h = bb.cpu().numpy().astype(np.int64).T
            size = (np.maximum(h, w) * 1.2).astype(np.int64)
            left = np.maximum(x + w / 2 - size / 2, 0).astype(np.int64)
            right = np.minimum(x + w / 2 + size / 2, 720).astype(np.int64)
            top = np.maximum(y + h / 2 - size / 2, 0).astype(np.int64)
            bottom = np.minimum(y + h / 2 + size / 2, 540).astype(np.int64)
            ci = torch.from_numpy(left[:, None] + cols[right - left]).to(r.device)
            ri = torch.from_numpy(top[:, None] + rows[bottom - top]).to(r.device)
            return bgr[vi, ri[:, :, None], ci[:, None, :]]

        ms_full, _ = timed(frames_then_crop)
        ms_fused, _ = timed(lambda: crops(0, m))
        same = torch.equal(frames_then_crop(), crops(0, m))
        lines.append("  %d views: full frames + crop %.1f ms (%.0f views/s); fused crops %.1f ms (%.0f views/s); identical crops: %s"
                     % (m, ms_full, m / ms_full * 1e3, ms_fused, m / ms_fused * 1e3, same))
        if label == "20k":
            ds_t = Dataset(None)
            np.random.seed(0)
            Rt, lt, ot = ds_t.training_draws(args.train)
            ms_train, _ = timed(lambda: r.render_crops_device(0, 720, 540, K, Rt, t, 10.0, 10000.0, lt, 1.2, 128, 128,
                                                              lights_y=fixed_light(), offsets=ot, want_mask=True, check=False))
            lines.append("  %d training pairs (x crop, mask, y crop): %.1f ms (%.0f pairs/s)" % (args.train, ms_train,
                                                                                                 args.train / ms_train * 1e3))
        r.close()
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        open(args.out, "w").write(text + "\n")


if __name__ == "__main__":
    main()
