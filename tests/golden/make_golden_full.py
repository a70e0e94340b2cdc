"""Generate tests/golden/ian_full_golden.npz: full IAN (reference IAN.py graph) oracle outputs on 2 CelebAValid
images + 2 random latents, synthetic seeded weights (see make_golden.py for the why).

    python tests/golden/make_golden_full.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ian_full_numpy as fn  # noqa: E402
from oracle import ian_numpy as on  # noqa: E402
from oracle import reference  # noqa: E402
from oracle import weights as ow  # noqa: E402

WEIGHT_SEED = 0
IDX = [420, 7]


def main():
    arr = np.load(os.path.join(reference.reference_dir(), 'CelebAValid.npz'))['arr_0']
    imgs = arr[IDX]
    P = ow.make_full_weights(WEIGHT_SEED)
    ordering = fn.made_ordering()
    masks = fn.made_masks(ordering)
    x = on.to_tanh(imgs.astype(np.float64)).astype(np.float32)
    mu, ls = fn.full_encode_mu_ls(P, x)
    z = fn.full_latent(P, mu, masks)
    rng = np.random.default_rng(11)
    eps = rng.standard_normal((2, 100)).astype(np.float32)
    z_sample = fn.full_latent(P, on.gaussian_sample(mu, ls, eps, deterministic=False), masks)
    xhat = fn.full_decode(P, z.astype(np.float32))
    z_rand = rng.standard_normal((2, 100)).astype(np.float32)
    xhat_rand = fn.full_decode(P, z_rand)
    out = os.path.join(ROOT, 'tests', 'golden', 'ian_full_golden.npz')
    np.savez_compressed(out, weight_seed=WEIGHT_SEED, idx=np.array(IDX), images=imgs, ordering=ordering.astype(np.int32),
                        mu=mu, logsigma=ls, z=z, eps=eps, z_sample=z_sample, xhat=xhat.astype(np.float32), z_rand=z_rand,
                        xhat_rand=xhat_rand.astype(np.float32))
    print('wrote', out, os.path.getsize(out), 'bytes')
    # ---- IANv1 (IANv1.py graph): same encoder/flow code path, different decoder
    Pv = ow.make_v1_weights(WEIGHT_SEED)
    mu1, ls1 = fn.full_encode_mu_ls(Pv, x)
    z1 = fn.full_latent(Pv, mu1, masks)
    xh1 = fn.v1_decode(Pv, z1.astype(np.float32))
    xr1 = fn.v1_decode(Pv, z_rand)
    out1 = os.path.join(ROOT, 'tests', 'golden', 'ian_v1_golden.npz')
    np.savez_compressed(out1, weight_seed=WEIGHT_SEED, images=imgs, ordering=ordering.astype(np.int32), mu=mu1, z=z1,
                        xhat=xh1.astype(np.float32), z_rand=z_rand, xhat_rand=xr1.astype(np.float32))
    print('wrote', out1, os.path.getsize(out1), 'bytes')


if __name__ == '__main__':
    main()
