"""GPU parity of the FULL IAN graph (reference IAN.py: MADE/IAF latent, MDC blocks, RGB-Beta head) through
API.IAN('IAN.py') -> C-ABI, against the float64 oracle's golden vectors.  Tolerances (float32 path):
  x_hat max-abs <= 2e-4 ; latents |dz| <= 3e-4 * (1 + |z|) (the IAF divides by exp(MADE_ls), |z| reaches ~10)."""
import os

import numpy as np
import pytest

from oracle import ian_full_numpy as fn
from oracle import ian_numpy as on
from oracle import weights as ow

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def gold():
    return dict(np.load(os.path.join(ROOT, "tests", "golden", "ian_full_golden.npz")))


@pytest.fixture(scope="module")
def PF(gold):
    return ow.make_full_weights(int(gold["weight_seed"]))


@pytest.fixture(scope="module")
def full_model(npe, PF):
    m = npe.IAN("IAN.py", dnn=True, weights=PF, device=0)
    yield m
    m.close()


@pytest.fixture(params=["tc", "simt"])
def fm(full_model, request):
    full_model.set_path(request.param)
    yield full_model
    full_model.set_path("tc")


def _zclose(z, ref, k=3e-4):
    return (np.abs(z - ref) <= k * (1.0 + np.abs(ref))).all()


def test_full_encode_golden(fm, gold):
    x = on.to_tanh(gold["images"].astype(np.float64)).astype(np.float32)
    z = fm.encode_images(x)
    assert z.shape == (2, 100) and _zclose(z, gold["z"]), np.abs(z - gold["z"]).max()
    zs = fm.encode(x, eps=gold["eps"])
    amp = np.abs(np.exp(gold["logsigma"]) * gold["eps"])
    assert (np.abs(zs - gold["z_sample"]) <= 1e-3 * (1.0 + np.abs(gold["z_sample"]) + amp)).all()


def test_full_decode_golden(fm, gold):
    xh = fm.sample_at(gold["z_rand"])
    assert xh.shape == (2, 3, 64, 64)
    assert np.abs(xh - gold["xhat_rand"]).max() <= 2e-4
    xh = fm.sample_at(gold["z"].astype(np.float32))
    assert np.abs(xh - gold["xhat"]).max() <= 2e-4


def test_full_reconstruct_and_ordering(full_model, gold, PF):
    assert np.array_equal(full_model.made_ordering, gold["ordering"])
    rng = np.random.default_rng(4)
    x = rng.uniform(-1, 1, (3, 3, 64, 64)).astype(np.float32)
    xh, z = full_model.reconstruct(x, return_z=True)
    masks = fn.made_masks(gold["ordering"].astype(np.float32))
    zr = fn.full_encode(PF, x[:1], masks)
    assert _zclose(z[:1], zr)
    assert np.abs(xh[:1] - fn.full_decode(PF, z[:1])).max() <= 2e-4
    assert np.abs(xh - full_model.sample_at(z)).max() <= 2e-4      # fused call vs two calls


def _rel(g, ref):
    return float(np.abs(g - ref).max() / np.abs(ref).max())


@pytest.mark.parametrize("which", ["v1", "full"])
@pytest.mark.parametrize("path", ["tc", "simt"])
def test_flow_model_brush_gradients(npe, which, path):
    """imgrad / imgradRGB (reference API.py:59,64,66-76) on the IANv1.py / IAN.py graphs: backward of the RGB-Beta head, the
    MDC residual blocks and the deconvs, against (a) numeric gradients of the EXECUTED reference (ref_exec_*.npz: g_light,
    g_rgb -- central differences of the reference's own forward) and (b) float64 autograd through the torch restatement on
    other samples / boxes.  Bound, as max-abs error / max|g|: <= 1e-3 on the executed-reference fixtures and on every batched
    case of IAN.py (LeakyRectify: measured <= 6e-4 tc, <= 4.5e-4 simt).  IANv1 is a ReLU network: a pre-activation within
    ~1e-5 of zero may fall on the other side of the rectifier than in float64 (activations carry 16 significand bits;
    tests/test_gpu_parity.py module docstring), and one such unit inside the brush footprint moves g by 0.3-1 %.
    tools/diag_flow_grad.py (profiles/r2_diag_flow_grad.log) shows it is per (sample, box) and hits BOTH CUDA paths, each on
    different cases, with everything else at 1e-5 -- so for IANv1 the batched bound is: every case <= 2e-2 and the unflipped
    cases (at least one of the six) <= 1e-4."""
    import json
    import torch
    from oracle import ian_torch as ot
    ref = np.load(os.path.join(ROOT, "tests", "golden", "ref_exec_%s.npz" % which))
    g0 = np.load(os.path.join(ROOT, "tests", "golden", "ian_%s_golden.npz" % which))
    Pn = (ow.make_v1_weights if which == "v1" else ow.make_full_weights)(int(g0["weight_seed"]))
    m = npe.IAN("IANv1.py" if which == "v1" else "IAN.py", True, weights=Pn, path=path)
    rec = {}
    try:
        c1, r1, c2, r2 = [int(v) for v in ref["grad_box"]]
        z = g0["z_rand"][:1].astype(np.float32)
        frame = np.broadcast_to(ref["grad_rgb_target"].astype(np.float32).reshape(1, 3, 1, 1), (1, 3, 64, 64)).copy()
        gl = m.imgrad(c1, r1, c2, r2, z)
        gr = m.imgradRGB(float(c1), float(r1), float(c2), float(r2), frame, z)       # NPE passes integral floats
        rec["fixture_light"], rec["fixture_rgb"] = _rel(gl, ref["g_light"]), _rel(gr, ref["g_rgb"])
        assert rec["fixture_light"] <= 1e-3 and rec["fixture_rgb"] <= 1e-3, rec
        # batched, per-sample boxes / colours, vs float64 autograd of the restatement
        P64 = ot.to_torch(Pn, torch.float64)
        dec = ot.v1_decode if which == "v1" else ot.full_decode
        rng = np.random.default_rng(8)
        zb = rng.standard_normal((3, 100)).astype(np.float32)
        boxes = np.array([[3, 5, 20, 17], [40, 30, 41, 31], [0, 47, 64, 64]], np.int32)
        rgb = rng.uniform(-1, 1, (3, 3)).astype(np.float32)
        g_rgb, g_light = m.grad(zb, boxes, rgb), m.grad(zb, boxes, None)
        for k in range(3):
            b = [int(v) for v in boxes[k]]
            zt = torch.from_numpy(zb[k:k + 1].astype(np.float64))
            fr = torch.from_numpy(np.broadcast_to(rgb[k].astype(np.float64).reshape(1, 3, 1, 1), (1, 3, 64, 64)).copy())
            rec["rgb_%d" % k] = _rel(g_rgb[k:k + 1], ot.imgradRGB(P64, b[0], b[1], b[2], b[3], fr, zt, decode_fn=dec).numpy())
            rec["light_%d" % k] = _rel(g_light[k:k + 1], ot.imgrad(P64, b[0], b[1], b[2], b[3], zt, decode_fn=dec).numpy())
        batched = [v for k, v in rec.items() if not k.startswith("fixture")]
        if which == "full":
            assert max(batched) <= 1e-3, rec
        else:
            assert max(batched) <= 2e-2 and min(batched) <= 1e-4, rec
        # the NPE step rule on this graph: two edit steps equal two manual gradient steps
        z2 = m.edit_steps(zb, boxes, rgb, n_steps=2, weight=0.05)
        zm = zb.copy()
        for _ in range(2):
            zm = (zm - np.float32(0.05) * m.grad(zm, boxes, rgb) * (1.0 + (boxes[:, 2] - boxes[:, 0]))[:, None]).astype(np.float32)
        assert np.abs(z2 - zm).max() <= 1e-5 * max(1.0, np.abs(zm).max())
    finally:
        m.close()
        if os.environ.get("IAN_TEST_RECORD"):
            os.makedirs(os.environ["IAN_TEST_RECORD"], exist_ok=True)
            with open(os.path.join(os.environ["IAN_TEST_RECORD"], "flow_brush_%s_%s.json" % (which, path)), "w") as f:
                json.dump(rec, f)


def test_custom_ordering_changes_masks(npe, PF):
    o = np.arange(100, dtype=np.int32)[::-1].copy()
    m = npe.IAN("IAN.py", True, weights=PF, made_ordering=o)
    rng = np.random.default_rng(5)
    x = rng.uniform(-1, 1, (1, 3, 64, 64)).astype(np.float32)
    z = m.encode_images(x)
    zr = fn.full_encode(PF, x, fn.made_masks(o.astype(np.float32)))
    m.close()
    assert _zclose(z, zr)
    with pytest.raises(npe.IanError):
        npe.IAN("IAN.py", True, weights=PF, made_ordering=np.zeros(100, np.int32))


def test_sample_ian_function_set(full_model, gold, PF):
    """sample / sampleZ / Zfn / Z_IAF_fn of reference sample_IAN.py:86-94."""
    x = on.to_tanh(gold["images"].astype(np.float64)).astype(np.float32)
    z0 = full_model.Zfn(x)
    assert np.abs(z0 - gold["mu"]).max() <= 2e-4
    z = full_model.Z_IAF_fn(gold["mu"].astype(np.float32))
    assert _zclose(z, gold["z"])
    xs = full_model.sample(gold["mu"].astype(np.float32))
    assert np.abs(xs - gold["xhat"]).max() <= 3e-4
    assert np.abs(full_model.sampleZ(gold["z_rand"]) - gold["xhat_rand"]).max() <= 2e-4
    grid = full_model.sample_grid(np.concatenate([x, x, x], 0), n_samples=3, seed=5)
    assert grid.shape == (3 + 3 * 9, 3, 64, 64) and np.isfinite(grid).all()
    assert np.array_equal(grid[3], x[0]) and np.array_equal(grid[3 + 8], x[1])     # endpoints bracket the interpolants


def test_simple_model_function_set_is_flowless(model, golden):
    x = on.to_tanh(golden["images"][:2].astype(np.float64)).astype(np.float32)
    assert np.abs(model.Zfn(x) - model.encode_images(x)).max() <= 2e-4     # same math through two entry points
    z = golden["z_rand"][:2]
    assert np.array_equal(model.Z_IAF_fn(z), z)
    assert np.abs(model.sample(z) - model.sample_at(z)).max() <= 5e-5


def test_bf16_mode_tolerance_vs_oracle(full_model, gold):
    """BASELINE configs[2]: full IAN in bf16 with an fp32 tolerance check.  Operands rounded to bf16 (8 significand
    bits), fp32 accumulation.  Measured on this fixture's [-1,1] images (final round-2 build; the kernels are
    deterministic, so every B200 gives these bits): max-abs 0.034 (the Beta ratio 2a/(a+b) is steep where both sigmoids
    are small), mean-abs 2.6e-3.  Bounds stated here: max-abs 0.08, mean-abs 5e-3 (bench.py reports max-abs / mean-abs /
    PSNR of bf16 vs float32 mode at batch 512: 0.065 / 2.8e-3 / 52.7 dB)."""
    x = on.to_tanh(gold["images"].astype(np.float64)).astype(np.float32)
    try:
        full_model.set_precision("bf16")
        xh = full_model.sample_at(gold["z_rand"])
        err = np.abs(xh - gold["xhat_rand"])
        print("bf16 vs oracle: max-abs %.4f mean-abs %.5f" % (err.max(), err.mean()))
        assert err.max() <= 0.08 and err.mean() <= 5e-3, (err.max(), err.mean())
        z = full_model.encode_images(x)
        assert (np.abs(z - gold["z"]) <= 6e-2 * (1.0 + np.abs(gold["z"]))).all()
        # the fp32 verification path run on the same bf16-rounded operands agrees to about the same level (bf16 re-rounding of activations amplifies 1-ulp differences)
        full_model.set_path("simt")
        xs = full_model.sample_at(gold["z_rand"])
        full_model.set_path("tc")
        assert np.abs(xs - xh).max() <= 0.1 and np.abs(xs - xh).mean() <= 5e-3, (np.abs(xs - xh).max(), np.abs(xs - xh).mean())
    finally:
        full_model.set_precision("fp32")
        full_model.set_path("tc")
    assert np.abs(full_model.sample_at(gold["z_rand"]) - gold["xhat_rand"]).max() <= 2e-4   # back to float32


def test_bf16_mode_is_full_model_only(model, npe):
    with pytest.raises(npe.IanError):
        model.set_precision("bf16")


# ---- IANv1.py graph -----------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def gold_v1():
    return dict(np.load(os.path.join(ROOT, "tests", "golden", "ian_v1_golden.npz")))


@pytest.mark.parametrize("path", ["tc", "simt"])
def test_ianv1_golden(npe, gold_v1, path):
    P1 = ow.make_v1_weights(int(gold_v1["weight_seed"]))
    m = npe.IAN("IANv1.py", dnn=True, weights=P1, path=path)
    try:
        x = on.to_tanh(gold_v1["images"].astype(np.float64)).astype(np.float32)
        z = m.encode_images(x)
        assert _zclose(z, gold_v1["z"]), np.abs(z - gold_v1["z"]).max()
        assert np.abs(m.Zfn(x) - gold_v1["mu"]).max() <= 2e-4
        xh = m.sample_at(gold_v1["z_rand"])
        assert np.abs(xh - gold_v1["xhat_rand"]).max() <= 2e-4
        assert np.abs(m.sample_at(gold_v1["z"].astype(np.float32)) - gold_v1["xhat"]).max() <= 2e-4
        if path == "tc":
            m.set_precision("bf16")
            err = np.abs(m.sample_at(gold_v1["z_rand"]) - gold_v1["xhat_rand"])
            print("IANv1 bf16 vs oracle: max-abs %.4f mean-abs %.5f" % (err.max(), err.mean()))
            assert err.max() <= 0.03 and err.mean() <= 3e-3     # measured 0.0061 / 7.5e-4 (plain deconv decoder: no steep MDC/Beta chain)
    finally:
        m.close()


@pytest.mark.parametrize("which", ["full", "v1"])
def test_pair_kernel_on_the_flow_models(npe, which, monkeypatch):
    """the CTA-pair tap-GEMM on the IAN.py / IANv1.py graphs (MDC taps, residual + raw-output epilogue of the MDBLOCKs),
    float32 split and single-pass bf16 mode, against the one-CTA kernel on the same schedule."""
    from oracle import weights as ow
    P = (ow.make_v1_weights if which == "v1" else ow.make_full_weights)(0)
    cfg = "IANv1.py" if which == "v1" else "IAN.py"
    for k, v in (("IAN_SPLITK", "0"), ("IAN_STREAMK", "0"), ("IAN_GRAPHS", "0")):
        monkeypatch.setenv(k, v)
    monkeypatch.setenv("IAN_TC2", "0")
    one = npe.IAN(cfg, True, weights=P)
    monkeypatch.setenv("IAN_TC2", "1")
    monkeypatch.setenv("IAN_TC2_MIN", "1")
    pair = npe.IAN(cfg, True, weights=P)
    rng = np.random.default_rng(43)
    try:
        for prec, tol in (("fp32", 1e-6), ("bf16", 1e-6)):
            one.set_precision(prec)
            pair.set_precision(prec)
            for n in (2, 5):
                x = rng.uniform(-1, 1, (n, 3, 64, 64)).astype(np.float32)
                xa, za = one.reconstruct(x, return_z=True)
                xb, zb = pair.reconstruct(x, return_z=True)
                assert np.abs(za - zb).max() <= tol and np.abs(xa - xb).max() <= tol, (prec, n)
    finally:
        one.close()
        pair.close()
