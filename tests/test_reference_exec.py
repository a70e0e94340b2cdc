"""The oracle against fixtures produced by EXECUTING the reference's own files (tests/golden/make_golden_ref.py):
API.IAN / IAN_simple.get_model / IANv1.get_model / IAN.get_model / layers.py / mask_generator.py /
GANcheckpoints.load_weights run unmodified from the reference checkout on numpy stand-ins for Theano and Lasagne
(oracle/refshim).  This is what pins the oracle: graph wiring, hyper-parameters, parameter names and the loading
path are the reference's code; only the third-party layer semantics underneath are restated.

The fixtures are float64 evaluations, so the float64 oracle must agree to rounding; the numeric gradients
(central differences of the reference forward) bound the analytic brush gradients."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import ian_full_numpy as fn
from oracle import ian_numpy as on
from oracle import reference
from oracle import weights as ow

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
DISCRIMINATOR = ["discrimi.W", "minibatch_discrim.b", "minibatch_discrim.log_weight_scale", "minibatch_discrim.theta"]


def _load(name):
    return np.load(os.path.join(GOLD, name))


def _names_match(ref, P):
    """the loader's parameter list (API.py:24-28) = the checkpoint contract: every name and shape"""
    want = {k: tuple(np.asarray(v).shape) for k, v in P.items() if k != "metadata"}
    got = {n: tuple(int(d) for d in s.split()) for n, s in zip(ref["param_names"], ref["param_shapes"])}
    assert sorted(set(got) - set(want)) == [n for n in DISCRIMINATOR if n not in want]     # heads we do not ship
    for n, shp in want.items():
        assert got[n] == shp, n


def test_simple_forward_matches_executed_reference(golden, weights):
    ref = dict(_load("ref_exec_simple.npz"), **_load("ref_exec_simple_rand.npz"))
    x = on.to_tanh(golden["images"].astype(np.float64)).astype(np.float32)
    mu, ls = on.simple_encode_mu_ls(weights, x)
    for tag, k in (("dnn", 8), ("nodnn", 2)):        # cuDNN GradI path and TransposedConv2D+Slice path are one function
        assert ref["mu_" + tag].shape == (k, 100)
        assert np.abs(mu[:k] - ref["mu_" + tag]).max() <= 1e-12
        assert np.abs(ls[:k] - ref["logsigma_" + tag]).max() <= 1e-12
        assert np.abs(on.simple_decode(weights, np.float32(ref["mu_" + tag])) - ref["xhat_" + tag]).max() <= 1e-12
        assert np.abs(on.simple_decode(weights, golden["z_rand"][:k]) - ref["xhat_rand_" + tag]).max() <= 1e-12
    assert np.abs(ref["xhat_dnn"][:2] - ref["xhat_nodnn"]).max() <= 1e-12
    _names_match(ref, weights)


def test_simple_gradients_match_numeric_gradients_of_executed_reference(golden, weights):
    """T.grad of API.py:59,64 evaluated as central differences (h=1e-6, float64) of the reference forward."""
    ref = _load("ref_exec_simple.npz")
    b = [int(v) for v in golden["boxes"][0]]
    frame = np.broadcast_to(golden["rgb"][0].reshape(1, 3, 1, 1), (1, 3, 64, 64)).astype(np.float32)
    cases = [(on.simple_imgradRGB(weights, b[0], b[1], b[2], b[3], frame, golden["z_rand"][:2]), ref["g0_rgb"]),
             (on.simple_imgrad(weights, b[0], b[1], b[2], b[3], golden["z_rand"][:2]), ref["g0_light"])]
    b5 = [int(v) for v in ref["g5_box"]]
    frame5 = np.broadcast_to(golden["rgb"][5].reshape(1, 3, 1, 1), (1, 3, 64, 64)).astype(np.float32)
    cases.append((on.simple_imgradRGB(weights, b5[0], b5[1], b5[2], b5[3], frame5, golden["z_rand"][5:6]), ref["g5_rgb"]))
    for mine, theirs in cases:
        assert mine.shape == theirs.shape
        assert np.abs(mine - theirs).max() <= 1e-6 * np.abs(theirs).max()      # measured 9e-9 (finite-difference accuracy)
    assert np.all(ref["g0_rgb"][1] == 0) and np.all(ref["g0_light"][1] == 0)  # the cost reads sample 0 only (API.py:59)


@pytest.mark.parametrize("which", ["v1", "full"])
def test_flow_models_match_executed_reference(which):
    ref = _load("ref_exec_%s.npz" % which)
    gold = _load("ian_%s_golden.npz" % which)
    P = (ow.make_v1_weights if which == "v1" else ow.make_full_weights)(int(gold["weight_seed"]))
    _names_match(ref, P)
    # MADE ordering and masks after reset("Once") (API.py:33-36)
    o = fn.made_ordering()
    assert np.array_equal(ref["ordering_mu"], o) and np.array_equal(ref["ordering_ls"], o)
    for mine, theirs in zip(fn.made_masks(o), (ref["mask_input"], ref["mask_output_W"], ref["mask_output_D"])):
        assert np.array_equal(mine, theirs)
    masks = fn.made_masks(o)
    x = on.to_tanh(gold["images"].astype(np.float64)).astype(np.float32)
    mu, ls = fn.full_encode_mu_ls(P, x)
    assert np.abs(mu - ref["mu"]).max() <= 1e-12 and np.abs(ls - ref["logsigma"]).max() <= 1e-12
    assert np.abs(fn.full_encode(P, x, masks) - ref["z"]).max() <= 1e-11
    assert np.abs(fn.full_latent(P, np.float32(ref["mu"]), masks) - ref["z_from_mu"]).max() <= 1e-11
    dec = fn.v1_decode if which == "v1" else fn.full_decode
    assert np.abs(dec(P, np.float32(ref["z"])) - ref["xhat"]).max() <= 1e-11
    assert np.abs(dec(P, gold["z_rand"]) - ref["xhat_rand"]).max() <= 1e-11
    assert np.abs(dec(P, fn.full_latent(P, gold["z_rand"], masks)) - ref["sample_rand"]).max() <= 1e-11   # sample_IAN.py:84


def test_made_layer_is_fed_its_own_input_layer():
    """the finding the executed reference forced on the oracle: inside the graph MADE sees relu(z W0 + b0), not z
    (layers.py:769 overwrites Layer.input_layer) -- a plain reading of MADE.get_output_for is measurably different."""
    ref = _load("ref_exec_v1.npz")
    gold = _load("ian_v1_golden.npz")
    P = ow.make_v1_weights(int(gold["weight_seed"]))
    masks = fn.made_masks(fn.made_ordering())
    z_iaf = np.float32(ref["mu"])
    as_read = fn.iaf(z_iaf, fn.made_core(P, "l_IAF_mu", z_iaf, masks), fn.made_core(P, "l_IAF_ls", z_iaf, masks))
    assert np.abs(as_read - ref["z_from_mu"]).max() > 0.1
    assert np.abs(fn.full_latent(P, z_iaf, masks) - ref["z_from_mu"]).max() <= 1e-11


@pytest.mark.skipif(reference.reference_dir() is None, reason="needs a checkout of ajbrock/Neural-Photo-Editor")
def test_fixture_regenerates_from_the_reference(tmp_path):
    """re-execute the reference (IANv1.py: encoder, MADE/IAF, decoder, RGB-Beta head) and compare with the committed file;
    the reference's sources are not part of this repository: oracle/reference.py says where its checkout is"""
    script = os.path.join(GOLD, "make_golden_ref.py")
    out = subprocess.run([sys.executable, script, "v1"], capture_output=True, text=True, timeout=600,
                         env=dict(os.environ, REF_EXEC_OUT=str(tmp_path), REF_EXEC_GRADS="0"))
    assert out.returncode == 0, out.stderr[-2000:]
    committed, fresh = _load("ref_exec_v1.npz"), np.load(tmp_path / "ref_exec_v1.npz")
    assert set(fresh.files) <= set(committed.files)          # the quick regeneration skips the numeric gradients
    for k in fresh.files:
        assert np.array_equal(committed[k], fresh[k]), k


def test_product_cfg_dicts_equal_the_reference_config_modules(npe):
    """API.IAN.cfg (reference API.py:18 reads it from the config module; NPE and sample_IAN.py read cfg['num_latents'])"""
    import json
    api = __import__(npe.__name__ + ".API", fromlist=["API"])
    norm = lambda v: {str(k): norm(x) for k, x in v.items()} if isinstance(v, dict) else (list(v) if isinstance(v, tuple) else v)
    for fixture, mine in (("ref_exec_v1.npz", dict(api._FULL_CFG, max_epochs=150)), ("ref_exec_full.npz", api._FULL_CFG),
                          ("ref_exec_simple.npz", api._SIMPLE_CFG)):
        ref = json.loads(str(_load(fixture)["cfg_json"]))
        keys = api._SIMPLE_MODEL_KEYS if fixture == "ref_exec_simple.npz" else api._FULL_MODEL_KEYS
        assert sorted(keys) == list(_load(fixture)["model_keys"])           # the dict get_model() returns (API.py:21)
        if fixture == "ref_exec_v1.npz":
            ref_wo, mine_wo = dict(ref), norm(mine)
            mine_wo.pop("ortho", None)                      # IANv1.py has no 'ortho' entry (API.py of the product pops it too)
            assert ref_wo == mine_wo
        else:
            assert ref == norm(mine), fixture


@pytest.mark.parametrize("which", ["v1", "full"])
def test_flow_model_brush_gradients_match_numeric_gradients_of_executed_reference(which):
    """oracle-only (the CUDA path has brush gradients for IAN_simple, DESIGN.md section 8): what API.py:59,64 would
    compute on the IANv1.py / IAN.py graphs -- autograd through the torch restatement vs central differences of the
    executed reference forward.  Ready-made target for the next scope row."""
    import torch
    from oracle import ian_torch as ot
    ref = _load("ref_exec_%s.npz" % which)
    gold = _load("ian_%s_golden.npz" % which)
    P = ot.to_torch((ow.make_v1_weights if which == "v1" else ow.make_full_weights)(int(gold["weight_seed"])), torch.float64)
    dec = ot.v1_decode if which == "v1" else ot.full_decode
    c1, r1, c2, r2 = [int(v) for v in ref["grad_box"]]
    z = torch.from_numpy(gold["z_rand"][:1].astype(np.float64))
    frame = torch.from_numpy(np.broadcast_to(ref["grad_rgb_target"].astype(np.float64).reshape(1, 3, 1, 1), (1, 3, 64, 64)).copy())
    g = ot.imgrad(P, c1, r1, c2, r2, z, decode_fn=dec).numpy()
    assert np.abs(g - ref["g_light"]).max() <= 1e-5 * np.abs(ref["g_light"]).max()
    g = ot.imgradRGB(P, c1, r1, c2, r2, frame, z, decode_fn=dec).numpy()
    assert np.abs(g - ref["g_rgb"]).max() <= 1e-5 * np.abs(ref["g_rgb"]).max()
