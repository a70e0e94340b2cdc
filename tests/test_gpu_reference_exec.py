"""The CUDA path against the fixtures produced by EXECUTING the reference (tests/golden/ref_exec_*.npz; see
tests/golden/make_golden_ref.py and tests/test_reference_exec.py) -- directly, not through the oracle.
Tolerances are the ones of test_gpu_parity.py / test_gpu_full.py (float32 semantics vs a float64 evaluation)."""
import os

import numpy as np
import pytest

from oracle import ian_numpy as on
from oracle import weights as ow

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ref(name):
    return np.load(os.path.join(ROOT, "tests", "golden", name))


def _zclose(z, ref, k=3e-4):
    return (np.abs(z - ref) <= k * (1.0 + np.abs(ref))).all()


@pytest.mark.parametrize("path", ["tc", "simt"])
def test_simple_against_executed_reference(model, golden, path):
    ref = _ref("ref_exec_simple.npz")
    model.set_path(path)
    try:
        x = on.to_tanh(golden["images"].astype(np.float64)).astype(np.float32)
        z = model.encode_images(x)                                        # API.IAN.encode_images (API.py:78-90)
        assert np.abs(z - ref["mu_dnn"]).max() <= 2e-4
        assert np.abs(model.sample_at(np.float32(ref["mu_dnn"])) - ref["xhat_dnn"]).max() <= 1e-4      # API.py:98-110
        assert np.abs(model.sample_at(golden["z_rand"]) - _ref("ref_exec_simple_rand.npz")["xhat_rand_dnn"]).max() <= 1e-4
        # brush gradients vs the numeric gradients of the reference forward (API.py:59,64)
        b = [int(v) for v in golden["boxes"][0]]
        frame = np.broadcast_to(golden["rgb"][0].reshape(1, 3, 1, 1), (1, 3, 64, 64)).astype(np.float32).copy()
        g = model.imgradRGB(b[0], b[1], b[2], b[3], frame, golden["z_rand"][:2])
        assert g.shape == (2, 100) and np.all(g[1] == 0)
        assert np.abs(g[0] - ref["g0_rgb"][0]).max() <= 1e-3 * np.abs(ref["g0_rgb"][0]).max()
        g = model.imgrad(b[0], b[1], b[2], b[3], golden["z_rand"][:2])
        assert np.abs(g[0] - ref["g0_light"][0]).max() <= 1e-3 * np.abs(ref["g0_light"][0]).max()
        b5 = [int(v) for v in ref["g5_box"]]
        frame5 = np.broadcast_to(golden["rgb"][5].reshape(1, 3, 1, 1), (1, 3, 64, 64)).astype(np.float32).copy()
        g = model.imgradRGB(b5[0], b5[1], b5[2], b5[3], frame5, golden["z_rand"][5:6])
        assert np.abs(g - ref["g5_rgb"]).max() <= 1e-3 * np.abs(ref["g5_rgb"]).max()
    finally:
        model.set_path("tc")


@pytest.mark.parametrize("which,config", [("v1", "IANv1.py"), ("full", "IAN.py")])
def test_flow_models_against_executed_reference(npe, which, config):
    ref = _ref("ref_exec_%s.npz" % which)
    gold = _ref("ian_%s_golden.npz" % which)
    P = (ow.make_v1_weights if which == "v1" else ow.make_full_weights)(int(gold["weight_seed"]))
    m = npe.IAN(config, dnn=True, weights=P)
    try:
        assert np.array_equal(m.made_ordering, ref["ordering_mu"].astype(np.int32))      # reset("Once"), API.py:33-36
        x = on.to_tanh(gold["images"].astype(np.float64)).astype(np.float32)
        for path in ("tc", "simt"):
            m.set_path(path)
            z = m.encode_images(x)                                        # Z_hat_fn: l_Z, through MADE + IAF
            assert _zclose(z, ref["z"]), np.abs(z - ref["z"]).max()
            assert np.abs(m.Zfn(x) - ref["mu"]).max() <= 2e-4             # sample_IAN.py:89
            assert _zclose(m.Z_IAF_fn(np.float32(ref["mu"])), ref["z_from_mu"])          # sample_IAN.py:92
            assert np.abs(m.sample_at(np.float32(ref["z"])) - ref["xhat"]).max() <= 2e-4
            assert np.abs(m.sample_at(gold["z_rand"]) - ref["xhat_rand"]).max() <= 2e-4
            assert np.abs(m.sample(gold["z_rand"]) - ref["sample_rand"]).max() <= 5e-4   # sample_IAN.py:84 (flow, then decode)
    finally:
        m.close()
