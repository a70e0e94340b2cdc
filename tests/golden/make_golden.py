"""Generate tests/golden/ian_simple_golden.npz.

Reads the reference's only real fixture, CelebAValid.npz (NPE.py:44), from its checkout (oracle/reference.py): picks 8
validation images (index 420 is NPE's default image) and pushes them through the
float64 oracle with SYNTHETIC seeded weights (the trained blobs are LFS pointers, SURVEY F2).
Tests read only the committed .npz.

    python tests/golden/make_golden.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ian_numpy as on  # noqa: E402
from oracle import reference  # noqa: E402
from oracle import weights as ow  # noqa: E402

WEIGHT_SEED = 0
IDX = [420, 0, 1, 2, 3, 500, 777, 999]


def main():
    arr = np.load(os.path.join(reference.reference_dir(), 'CelebAValid.npz'))['arr_0']
    assert arr.shape == (1000, 3, 64, 64) and arr.dtype == np.uint8
    imgs = arr[IDX]
    P = ow.make_simple_weights(WEIGHT_SEED)
    x = on.to_tanh(imgs.astype(np.float64)).astype(np.float32)       # NPE.py:257 passes float32
    mu, ls = on.simple_encode_mu_ls(P, x)
    rng = np.random.default_rng(7)
    eps = rng.standard_normal((8, 100)).astype(np.float32)
    z_sample = on.gaussian_sample(mu, ls, eps, deterministic=False)
    xhat = on.simple_decode(P, mu.astype(np.float32))
    z_rand = rng.standard_normal((8, 100)).astype(np.float32)
    xhat_rand = on.simple_decode(P, z_rand)
    # brush gradients: NPE-law boxes (side 1..17 inside the frame, NPE.py:149-156)
    side = rng.integers(1, 18, size=8)
    c1 = np.array([rng.integers(0, 64 - s + 1) for s in side])
    r1 = np.array([rng.integers(0, 64 - s + 1) for s in side])
    boxes = np.stack([c1, r1, c1 + side, r1 + side], 1).astype(np.int32)
    rgb = rng.uniform(-1, 1, (8, 3)).astype(np.float32)
    g_rgb = on.simple_grad_batched(P, z_rand, boxes, rgb)
    g_light = on.simple_grad_batched(P, z_rand, boxes, None)
    # single-sample API forms on sample 0 with a full-frame RGB target (NPE.py:205)
    frame = np.broadcast_to(rgb[0].reshape(1, 3, 1, 1), (1, 3, 64, 64)).astype(np.float32)
    g0_rgb = on.simple_imgradRGB(P, boxes[0, 0], boxes[0, 1], boxes[0, 2], boxes[0, 3], frame, z_rand[:2])
    g0_light = on.simple_imgrad(P, float(boxes[0, 0]), float(boxes[0, 1]), float(boxes[0, 2]), float(boxes[0, 3]), z_rand[:2])
    # short edit loop (4 samples x 4 steps, float32 state)
    z_edit = on.simple_edit_loop(P, z_rand[:4], boxes[:4], rgb[:4], n_steps=4, weight=0.05)
    out = os.path.join(ROOT, 'tests', 'golden', 'ian_simple_golden.npz')
    np.savez_compressed(out, weight_seed=WEIGHT_SEED, idx=np.array(IDX), images=imgs, mu=mu, logsigma=ls, eps=eps,
                        z_sample=z_sample, xhat=xhat.astype(np.float32), z_rand=z_rand,
                        xhat_rand=xhat_rand.astype(np.float32), boxes=boxes, rgb=rgb, g_rgb=g_rgb, g_light=g_light,
                        g0_rgb=g0_rgb, g0_light=g0_light, z_edit=z_edit)
    print('wrote', out, os.path.getsize(out), 'bytes')


if __name__ == '__main__':
    main()
