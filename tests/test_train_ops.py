"""Training-mode pieces (SURVEY 8f rank 4): BatchNorm with batch statistics and the MinibatchLayer forward.

CPU part: the float64 oracle (oracle/train_numpy.py) against tests/golden/ref_exec_train.npz -- the reference's own
MinibatchLayer class executed from the reference checkout, and lasagne's training-mode batch_norm through the stand-in.
GPU part: the CUDA ops through the C-ABI against the same fixture and against the oracle at training-size shapes
(batch 128 conv activations; the 16384 -> 100x5 minibatch discrimination of IAN_simple.py:225-231).
Tolerance: 2e-5 relative to the output scale (float32 data, float64-accumulated statistics)."""
import importlib
import os

import numpy as np
import pytest

from oracle import train_numpy as tn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = np.load(os.path.join(ROOT, "tests", "golden", "ref_exec_train.npz"))


def test_oracle_matches_the_executed_reference_minibatch_layer():
    out = tn.minibatch_layer(REF["mb_x"], REF["mb_theta"], REF["mb_lws"], REF["mb_b"])
    assert out.shape == REF["mb_out"].shape == (6, 64 + 7)
    assert np.abs(out - REF["mb_out"]).max() <= 1e-12
    assert np.array_equal(out[:, :64], REF["mb_x"].reshape(6, -1).astype(np.float64))     # concat([input, f])


def test_oracle_matches_training_mode_batch_norm():
    for tag in ("conv", "dense"):
        x = REF["bn_%s_x" % tag]
        c = x.shape[1]
        y, rm, ris, mean, inv_std = tn.batch_norm_train(x, REF["bn_%s_gamma" % tag], REF["bn_%s_beta" % tag], np.zeros(c), np.ones(c))
        assert np.abs(y - REF["bn_%s_y" % tag]).max() <= 1e-12
        axes = (0,) + tuple(range(2, x.ndim))
        assert np.allclose(rm, 0.1 * x.astype(np.float64).mean(axes)) and np.allclose(ris, 0.9 + 0.1 * inv_std)
        yn = (y - REF["bn_%s_beta" % tag].reshape([1, -1] + [1] * (x.ndim - 2))) / REF["bn_%s_gamma" % tag].reshape([1, -1] + [1] * (x.ndim - 2))
        assert np.abs(yn.mean(axes)).max() <= 1e-9 and np.abs(yn.var(axes) - 1).max() <= 1e-3   # eps = 1e-4 inside the sqrt


@pytest.mark.gpu
def test_gpu_batch_norm_train_and_minibatch_layer(model):
    import torch
    ops = importlib.import_module("neural-photo-editor_b200.train_ops")
    dev = torch.device("cuda", 0)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
    # fixture shapes (executed reference)
    for tag in ("conv", "dense"):
        x = REF["bn_%s_x" % tag]
        c = x.shape[1]
        rm, ris = t(np.full(c, 0.25)), t(np.full(c, 1.5))
        y = ops.batch_norm_train(model, t(x), t(REF["bn_%s_gamma" % tag]), t(REF["bn_%s_beta" % tag]), rm, ris)
        torch.cuda.synchronize()
        assert np.abs(y.cpu().numpy() - REF["bn_%s_y" % tag]).max() <= 2e-5
        _, rm_ref, ris_ref, _, _ = tn.batch_norm_train(x, REF["bn_%s_gamma" % tag], REF["bn_%s_beta" % tag], np.full(c, 0.25), np.full(c, 1.5))
        assert np.abs(rm.cpu().numpy() - rm_ref).max() <= 1e-6 and np.abs(ris.cpu().numpy() - ris_ref).max() <= 1e-5
    out = ops.minibatch_layer(model, t(REF["mb_x"]), t(REF["mb_theta"]), t(REF["mb_lws"]), t(REF["mb_b"]))
    torch.cuda.synchronize()
    assert np.abs(out.cpu().numpy() - REF["mb_out"]).max() <= 2e-5
    # training-size shapes: bnorm2 of IAN_simple (batch 128, 256 x 16 x 16), a dense BN (128 x 1000), the discriminator's
    # minibatch features (16384 -> 100 kernels x 5)
    rng = np.random.default_rng(3)
    for shape in ((128, 256, 16, 16), (128, 1000), (3, 8, 5, 7)):
        x = (rng.standard_normal(shape) * 1.7 + 0.3).astype(np.float32)
        c = shape[1]
        g, b = rng.uniform(0.5, 1.5, c).astype(np.float32), rng.normal(0, 0.1, c).astype(np.float32)
        rm0, ris0 = rng.normal(0, 0.1, c).astype(np.float32), rng.uniform(0.5, 2, c).astype(np.float32)
        rm, ris = t(rm0), t(ris0)
        y = ops.batch_norm_train(model, t(x), t(g), t(b), rm, ris)
        y2 = ops.batch_norm_train(model, t(x), t(g), t(b))                 # no running statistics: same y, bit for bit
        torch.cuda.synchronize()
        y_ref, rm_ref, ris_ref, _, _ = tn.batch_norm_train(x, g, b, rm0, ris0)
        assert np.abs(y.cpu().numpy() - y_ref).max() <= 2e-5 * max(1.0, np.abs(y_ref).max()), shape
        assert torch.equal(y, y2)
        assert np.abs(rm.cpu().numpy() - rm_ref).max() <= 1e-6 and np.abs(ris.cpu().numpy() - ris_ref).max() <= 1e-5
    x = rng.standard_normal((32, 1024, 4, 4)).astype(np.float32) * 0.5
    theta = rng.normal(0, 0.05, (16384, 100, 5)).astype(np.float32)
    lws, b = rng.normal(0, 0.2, (100, 5)).astype(np.float32), np.full(100, -1.0, np.float32)
    out = ops.minibatch_layer(model, t(x), t(theta), t(lws), t(b))
    torch.cuda.synchronize()
    ref = tn.minibatch_layer(x, theta, lws, b)
    assert out.shape == (32, 16384 + 100)
    assert np.abs(out.cpu().numpy() - ref).max() <= 2e-5 * max(1.0, np.abs(ref).max())
