"""Plat-style model API of the Neural Photo Editor, backed by libian_b200.so (sm_100a CUDA).

Drop-in for the reference `API.py` (reference API.py:11-110): same class name, constructor signature
and method surface (`encode_images`, `sample_at`, `get_zdim`, `imgrad`, `imgradRGB`, attributes `cfg`,
`weights_fname`, `model`), so `NPE.py:18  model = IAN(config_path='IAN_simple.py', dnn=True)` and every
later call in NPE.py work unchanged.  All numerics run in the CUDA library through its C-ABI
(include/ian_b200.h); this file only marshals numpy arrays.  There is no Theano/Lasagne dependency and
no CPU fallback.

Extensions beyond the reference surface (SURVEY.md section 8b): `reconstruct`, `encode(..., eps)`,
batched `grad` / `edit_steps`, and `*_dev` variants taking device pointers.
"""
from __future__ import annotations

import ctypes as C
import os
import warnings

import numpy as np

from . import _lib

# cfg of reference IAN_simple.py:33-51 (the config module itself imports lasagne/theano and cannot
# be executed here; the hot path only reads cfg['num_latents'], API.py:96)
_SIMPLE_CFG = {
    'batch_size': 128, 'learning_rate': {0: 0.0002}, 'optimizer': 'Adam', 'beta1': 0.5, 'update_ratio': 1,
    'decay_rate': 0, 'reg': 1e-5, 'momentum': 0.9, 'shuffle': True, 'dims': (64, 64), 'n_channels': 3,
    'n_classes': 10, 'batches_per_chunk': 64, 'max_epochs': 250, 'checkpoint_every_nth': 1, 'num_latents': 100,
    'recon_weight': 3.0, 'feature_weight': 1.0,
}
_SIMPLE_MODEL_KEYS = ('l_in', 'l_out', 'l_mu', 'l_ls', 'l_Z', 'l_introspect', 'l_discrim')
# cfg of reference IAN.py:39-62
_FULL_CFG = {
    'batch_size': 16, 'learning_rate': {0: 0.0002, 25: 0.0001, 50: 0.00005, 75: 0.00001}, 'optimizer': 'Adam',
    'beta1': 0.5, 'update_ratio': 1, 'decay_rate': 0, 'reg': 1e-5, 'momentum': 0.9, 'shuffle': True, 'dims': (64, 64),
    'n_channels': 3, 'batches_per_chunk': 64, 'max_epochs': 80, 'checkpoint_every_nth': 1, 'num_latents': 100,
    'recon_weight': 3.0, 'feature_weight': 1.0, 'dg_weight': 1.0, 'dd_weight': 1.0, 'agr_weight': 1.0,
    'ags_weight': 1.0, 'n_shuffles': 1, 'ortho': 1e-3,
}
_FULL_MODEL_KEYS = _SIMPLE_MODEL_KEYS + ('l_IAF_mu', 'l_IAF_ls', 'l_Z_IAF')


def made_ordering(seed=1234, n=100):
    """MADE input ordering after `reset("Once")` (reference API.py:33-36 -> layers.py:845-853 ->
    mask_generator.py:35-38,55-73): one shuffle_row_elements draw of theano RandomStreams(seed).  Recalled theano
    seeding (SURVEY Appendix D, unverifiable offline): the stream's generator is
    RandomState(RandomState(seed).randint(2**30)) and a 1-D shuffle is one permutation(n).  Pass
    `made_ordering=` to IAN(...) to override."""
    stream = np.random.RandomState(int(np.random.RandomState(seed).randint(2 ** 30)))
    return np.arange(n, dtype=np.int32)[stream.permutation(n)]


def _f32(a, ndim, what):
    """theano.function input filtering for a float32 TensorType: wrong dtype / ndim -> TypeError."""
    a = np.asarray(a)
    if a.dtype != np.float32:
        raise TypeError("%s must be float32 (got %s); the reference's theano function rejects it too" % (what, a.dtype))
    if a.ndim != ndim:
        raise TypeError("%s must have %d dimensions (got %d)" % (what, ndim, a.ndim))
    return np.ascontiguousarray(a)


def _int_scalar(v, what):
    """int32 scalar input: non-integral values are rejected, integral floats accepted (NPE.py:202 passes
    `coords//4` floats); assumption C.8 in SURVEY.md."""
    iv = int(v)
    if iv != v:
        raise TypeError("%s=%r is not an integral value" % (what, v))
    return iv


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _z(a, what='z'):
    """latents: float32 (n,100).  The C side assumes the trailing dimension; theano would raise a shape error."""
    a = _f32(a, 2, what)
    if a.shape[1] != 100:
        raise ValueError("%s must be (n,100), got %r" % (what, a.shape))
    return a


def _img(a, what='images'):
    """images: float32 (n,3,64,64) NCHW."""
    a = _f32(a, 4, what)
    if a.shape[1:] != (3, 64, 64):
        raise ValueError("%s must be (n,3,64,64), got %r" % (what, a.shape))
    return a


def model_param_specs(kind):
    """[(name, shape)] of the graph's own parameters, in the reference's checkpoint naming -- the list API.py:23-28
    builds with lasagne.layers.get_all_params and hands to GANcheckpoints.load_weights."""
    lib = _lib.load()
    n = lib.ian_model_param_count(int(kind))
    if n < 0:
        raise ValueError("unknown model kind %r" % (kind,))
    out = []
    for i in range(n):
        name, shape, nd = C.c_char_p(), (C.c_int64 * 4)(), C.c_int()
        if lib.ian_model_param_spec(int(kind), i, C.byref(name), shape, C.byref(nd)) != _lib.IAN_OK:
            raise RuntimeError("ian_model_param_spec(%d, %d) failed" % (kind, i))
        out.append((name.value.decode(), tuple(int(shape[k]) for k in range(nd.value))))
    return out


class IAN:
    """Generic class for using IAN style models with the NPE (reference API.py:11)."""

    def __init__(self, config_path, dnn=True, weights=None, device=0, path=None, made_ordering=None):
        """config_path: path of the reference-style config module ('IAN_simple.py'); the weights are read
        from config_path[:-3]+'.npz' in GANcheckpoints format (reference API.py:18-30) unless a
        {name: ndarray} dict is given in `weights`.  `dnn` is accepted for signature compatibility (both
        reference variants of the graph are numerically the same function, IAN_simple.py:141-223)."""
        base = os.path.basename(str(config_path))
        if base == 'IAN_simple.py':
            kind, self.cfg, keys = _lib.IAN_MODEL_SIMPLE, dict(_SIMPLE_CFG), _SIMPLE_MODEL_KEYS
        elif base == 'IAN.py':
            # the reference's own API.IAN cannot construct this config (get_model(interp=...) vs dnn=..., SURVEY F6)
            kind, self.cfg, keys = _lib.IAN_MODEL_FULL, dict(_FULL_CFG), _FULL_MODEL_KEYS
        elif base == 'IANv1.py':
            kind, self.cfg, keys = _lib.IAN_MODEL_V1, dict(_FULL_CFG, max_epochs=150), _FULL_MODEL_KEYS
            self.cfg.pop('ortho', None)                     # IANv1.py:39-61 has no 'ortho' entry
        else:
            raise NotImplementedError("config %r: known graphs are IAN_simple.py, IAN.py and IANv1.py" % base)
        self.kind = kind
        self.weights_fname = str(config_path)[:-3] + '.npz'
        self.model = {k: base[:-3] + '.' + k for k in keys}
        self.dnn = dnn
        self._lib = _lib.load()
        self._stream_outs = {}                              # reconstruct_stream's rotating pinned result buffers
        self._h = C.c_void_p()
        rc = self._lib.ian_create(kind, int(device), C.byref(self._h))
        if rc != _lib.IAN_OK:
            msg = self._lib.ian_last_error(None)
            self._h = None
            raise _lib.IanError("ian_create failed (%d): %s" % (rc, msg.decode() if msg else "?"))
        print('Loading weights')
        if weights is None:
            weights = np.load(self.weights_fname, allow_pickle=False)
        # GANcheckpoints.load_weights (reference GANcheckpoints.py:33-57): iterate the MODEL's parameters and look each
        # one up by name; keys of the file the graph does not own (the trainer's log_sigma_theta,
        # train_IAN_simple.py:300,564; discriminator weights; the pickled 'metadata') are ignored.  Where the reference
        # only warns -- a parameter missing from the file, a shape mismatch -- this loader raises (ian_set_param /
        # ian_finalize), because a silently half-loaded model is never what a caller wants.
        have = set(weights.keys() if hasattr(weights, 'keys') else weights)
        own = model_param_specs(kind)
        for name, _shape in own:
            if name not in have:
                continue                                    # reported by ian_finalize as "missing parameter"
            arr = np.ascontiguousarray(np.asarray(weights[name], dtype=np.float32))
            shape = (C.c_int64 * max(arr.ndim, 1))(*arr.shape)
            self._check(self._lib.ian_set_param(self._h, name.encode(), _fp(arr), shape, arr.ndim))
        self.ignored_keys = sorted(have - {n for n, _ in own})
        if kind != _lib.IAN_MODEL_SIMPLE:
            print('Shuffling MADE masks')                   # reference API.py:33-36
            o = np.ascontiguousarray(globals()['made_ordering']() if made_ordering is None else made_ordering, np.int32)
            self.made_ordering = o
            self._check(self._lib.ian_set_made_ordering(self._h, o.ctypes.data_as(C.POINTER(C.c_int32)), int(o.size)))
        self._check(self._lib.ian_finalize(self._h))
        if path is not None:
            self.set_path(path)

    # ---- plumbing ---------------------------------------------------------------------------
    def _check(self, rc):
        _lib.check(self._lib, self._h, rc)

    def close(self):
        if getattr(self, '_h', None):
            self._lib.ian_destroy(self._h)
            self._h = None
            self._stream_outs = {}                          # the pinned memory went with the handle

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_path(self, path):
        """'tc' (tcgen05, default) or 'simt' (fp32 FFMA verification path); both are CUDA."""
        self._check(self._lib.ian_set_path(self._h, {'tc': _lib.IAN_PATH_TC, 'simt': _lib.IAN_PATH_SIMT}[path]))

    def set_precision(self, precision):
        """'fp32' (default: float32 semantics via the 3-pass bf16 split) or 'bf16' (full IAN only, single pass)."""
        self._check(self._lib.ian_set_precision(self._h, {'fp32': 0, 'bf16': 1}[precision]))

    def launch_count(self):
        return int(self._lib.ian_launch_count(self._h))

    def set_layer_timing(self, enable):
        self._check(self._lib.ian_set_layer_timing(self._h, int(bool(enable))))

    def layer_time_ms(self, layer, reset=True):
        return float(self._lib.ian_layer_time_ms(self._h, layer.encode(), int(reset)))

    # ---- reference surface ------------------------------------------------------------------------
    def imgrad(self, c1, r1, c2, r2, z):
        """Change in latents which would lighten the local image patch (reference API.py:66-70)."""
        return self._imgrad(c1, r1, c2, r2, None, z)

    def imgradRGB(self, c1, r1, c2, r2, RGB, z):
        """Change in latents which would move the local patch towards RGB (reference API.py:72-76)."""
        return self._imgrad(c1, r1, c2, r2, RGB, z)

    def _imgrad(self, c1, r1, c2, r2, RGB, z):
        c1, r1, c2, r2 = (_int_scalar(v, n) for v, n in zip((c1, r1, c2, r2), ('c1', 'r1', 'c2', 'r2')))
        z = _z(z)
        out = np.zeros_like(z)        # only sample 0 is differentiated (API.py:59,64)
        if z.shape[0] == 0:
            return out
        # numpy/theano slice semantics of X_hat[0,:,r1:r2,c1:c2]
        ra, rb, _ = slice(r1, r2).indices(64)
        ca, cb, _ = slice(c1, c2).indices(64)
        if rb <= ra or cb <= ca:
            out[0] = np.nan           # mean over an empty slice (cannot occur from NPE.py:149)
            return out
        boxes = np.array([[ca, ra, cb, rb]], dtype=np.int32)
        tgt = None
        if RGB is not None:
            RGB = _f32(RGB, 4, 'RGB')
            tgt = np.ascontiguousarray(RGB[0:1])
            if tgt.shape != (1, 3, 64, 64):
                raise TypeError("RGB must be (>=1,3,64,64), got %r" % (RGB.shape,))
        g = np.empty((1, z.shape[1]), np.float32)
        self._check(self._lib.ian_grad_host(self._h, _fp(np.ascontiguousarray(z[0:1])),
                                            boxes.ctypes.data_as(C.POINTER(C.c_int32)),
                                            _fp(tgt) if tgt is not None else None, 1, 1, _fp(g)))
        out[0] = g[0]
        return out

    def encode_images(self, images):
        """Encode images x => z: (n,3,s,s) float32 in [-1,1] -> (n, zdim) (reference API.py:78-90)."""
        return self.encode(images)

    def get_zdim(self):
        """Integer dimension of the latent z space (reference API.py:92-96)."""
        return self.cfg['num_latents']

    def sample_at(self, z):
        """Decode images z => x: (n, zdim) float32 -> (n,3,s,s) in [-1,1] (reference API.py:98-110)."""
        z = _z(z)
        x = np.empty((z.shape[0], 3, 64, 64), np.float32)
        if z.shape[0]:
            self._check(self._lib.ian_decode_host(self._h, _fp(z), z.shape[0], _fp(x)))
        return x

    # ---- extensions (batched / reparameterised / fused) ------------------------------------------
    def encode(self, images, eps=None):
        """deterministic (eps=None): mu(x).  With eps (n,100): mu + exp(logsigma)*eps (layers.py:419-433)."""
        x = _img(images)
        n = x.shape[0]
        z = np.empty((n, 100), np.float32)
        if n:
            e = None if eps is None else _z(eps, 'eps')
            if e is not None and e.shape[0] != n:
                raise ValueError("eps must be (%d,100), got %r" % (n, e.shape))
            self._check(self._lib.ian_encode_host(self._h, _fp(x), n, _fp(e) if e is not None else None, _fp(z)))
        return z

    # ---- the reference sampling script's function set (sample_IAN.py:86-94) ---------------------------------
    def Zfn(self, images):
        """X -> l_Z_IAF, deterministic (= mu, before the MADE/IAF flow); sample_IAN.py:91."""
        x = _img(images)
        z = np.empty((x.shape[0], 100), np.float32)
        if x.shape[0]:
            self._check(self._lib.ian_encode_pre_host(self._h, _fp(x), x.shape[0], _fp(z)))
        return z

    def Z_IAF_fn(self, z_iaf):
        """l_Z_IAF -> l_Z through the MADE/IAF flow (identity for IAN_simple); sample_IAN.py:94."""
        z0 = _z(z_iaf)
        z = np.empty_like(z0)
        if z0.shape[0]:
            self._check(self._lib.ian_flow_host(self._h, _fp(z0), z0.shape[0], _fp(z), None))
        return z

    def sample(self, z_iaf):
        """l_Z_IAF -> X: flow, then decoder; sample_IAN.py:86 (what the script feeds N(0,1) noise to)."""
        z0 = _z(z_iaf)
        x = np.empty((z0.shape[0], 3, 64, 64), np.float32)
        if z0.shape[0]:
            self._check(self._lib.ian_flow_host(self._h, _fp(z0), z0.shape[0], None, _fp(x)))
        return x

    def sampleZ(self, z):
        """l_Z -> X; sample_IAN.py:88 (== sample_at)."""
        return self.sample_at(z)

    def sample_grid(self, endpoints, n_samples=27, seed=None):
        """The 6x9 grid of sample_IAN.py:173-187: n_samples random samples + 3 rows of [endpoint, 7 interpolants,
        endpoint].  `endpoints`: 6 images float32 (6,3,64,64) in [-1,1].  Returns float32 images in [-1,1]."""
        rng = np.random.RandomState(seed)
        samples = self.sample(rng.randn(n_samples, 100).astype(np.float32))
        ends = _img(endpoints, 'endpoints')
        Ze = self.Zfn(ends)
        Z = np.asarray([Ze[2 * i] * (1 - j) + Ze[2 * i + 1] * j for i in range(3) for j in [t / 6.0 for t in range(7)]],
                       dtype=np.float32)
        rows = [np.insert(ends[2 * i:2 * (i + 1)], 1, self.sample(Z[7 * i:7 * (i + 1)]), axis=0) for i in range(3)]
        return np.append(samples, np.concatenate(rows, axis=0), axis=0)

    def reconstruct(self, images, return_z=False, out=None):
        """encode -> decode in one library call (the BASELINE metric's path).  `out`: optional preallocated
        float32 (n,3,64,64) result buffer (e.g. from pinned_empty) to avoid a pageable allocation per call."""
        x = _img(images)
        n = x.shape[0]
        xh = np.empty_like(x) if out is None else self._out(out, x.shape)
        z = np.empty((n, 100), np.float32)
        if n:
            self._check(self._lib.ian_reconstruct_host(self._h, _fp(x), n, _fp(z), _fp(xh)))
        return (xh, z) if return_z else xh

    @staticmethod
    def _out(out, shape):
        if not (isinstance(out, np.ndarray) and out.dtype == np.float32 and out.shape == tuple(shape)
                and out.flags['C_CONTIGUOUS']):
            raise TypeError("out must be a C-contiguous float32 array of shape %r" % (tuple(shape),))
        return out

    def pinned_empty(self, shape):
        """float32 numpy array in page-locked host memory owned by this model (valid until close())."""
        nbytes = int(np.prod(shape)) * 4
        p = C.c_void_p()
        self._check(self._lib.ian_host_alloc(self._h, nbytes, C.byref(p)))
        buf = (C.c_float * (nbytes // 4)).from_address(p.value)
        return np.frombuffer(buf, dtype=np.float32).reshape(shape)

    def reconstruct_submit(self, images, out, z_out=None):
        """Pipelined encode -> decode: enqueue one batch (n <= 512) and return a ticket immediately; `out`
        (and `z_out`) receive the result once reconstruct_wait(ticket) returns.  Two requests may be in
        flight; use pinned_empty() buffers so the copies overlap the neighbouring requests' compute."""
        x = _img(images)
        n = x.shape[0]
        out = self._out(out, x.shape)
        if z_out is not None:
            z_out = self._out(z_out, (n, 100))
        t = C.c_int()
        self._check(self._lib.ian_reconstruct_submit(self._h, _fp(x), n, _fp(z_out) if z_out is not None else None,
                                                     _fp(out), C.byref(t)))
        return t.value

    def reconstruct_wait(self, ticket):
        self._check(self._lib.ian_reconstruct_wait(self._h, int(ticket)))

    def reconstruct_stream(self, batches):
        """Generator over an iterable of (n,3,64,64) float32 batches: yields each reconstruction in order while
        keeping two batches in flight (H2D / compute / D2H of neighbouring batches overlap).  The yielded array
        is one of two rotating pinned buffers owned by the model (allocated on first use per batch shape, reused by
        later calls): consume it before advancing the generator twice, and run one stream at a time."""
        outs, pending = self._stream_outs, None              # page-locking costs milliseconds: keep the buffers
        for i, x in enumerate(batches):
            x = _img(x)
            key = (i & 1, x.shape)
            if key not in outs:
                outs[key] = self.pinned_empty(x.shape)
            t = self.reconstruct_submit(x, outs[key])
            if pending is not None:
                self.reconstruct_wait(pending[0])
                yield pending[1]
            pending = (t, outs[key])
        if pending is not None:
            self.reconstruct_wait(pending[0])
            yield pending[1]

    def _target(self, rgb, n):
        if rgb is None:
            return None, 0
        rgb = _f32(rgb, np.asarray(rgb).ndim, 'rgb')
        if rgb.shape == (n, 3):
            return rgb, 0
        if rgb.shape == (n, 3, 64, 64):
            return rgb, 1
        raise ValueError("rgb must be (n,3) or (n,3,64,64), got %r" % (rgb.shape,))

    def grad(self, z, boxes, rgb=None):
        """Per-sample brush gradient: boxes (n,4) int32 [c1,r1,c2,r2]; rgb None (lighten), (n,3) or frames."""
        z = _z(z)
        n = z.shape[0]
        boxes = np.ascontiguousarray(np.asarray(boxes, dtype=np.int32).reshape(n, 4))
        t, is_frame = self._target(rgb, n)
        g = np.empty_like(z)
        self._check(self._lib.ian_grad_host(self._h, _fp(z), boxes.ctypes.data_as(C.POINTER(C.c_int32)),
                                            _fp(t) if t is not None else None, is_frame, n, _fp(g)))
        return g

    def edit_steps(self, z, boxes, rgb=None, n_steps=32, weight=0.05):
        """n_steps of the NPE paint rule per sample: Z <- Z - weight*g*(1+(x2-x1)) (reference NPE.py:199-209)."""
        z = _z(z).copy()
        n = z.shape[0]
        boxes = np.ascontiguousarray(np.asarray(boxes, dtype=np.int32).reshape(n, 4))
        t, is_frame = self._target(rgb, n)
        self._check(self._lib.ian_edit_loop_host(self._h, _fp(z), boxes.ctypes.data_as(C.POINTER(C.c_int32)),
                                                 _fp(t) if t is not None else None, is_frame, n, int(n_steps),
                                                 float(weight)))
        return z

    def paint_stroke(self, z, box, rgb_frame, recon_u8, error, weight=0.05):
        """One NPE paint stroke in photo mode in a single library call (reference NPE.py:199-231): brush gradient,
        latent update, re-decode, DELTA/MASK(gaussian 0.7)/ERROR blend, uint8 conversion and the 4x display upsample.
        z (1,100) float32; box = (x1,y1,x2,y2) as NPE computes it (integral floats accepted); rgb_frame (1,3,64,64)
        float32 = to_tanh(myRGB); recon_u8 (3,64,64) uint8; error (3,64,64) float32.
        Returns (z_new (1,100), IM uint8 (3,64,64), display uint8 (256,256,3) ready for PIL.Image.fromarray)."""
        z = _f32(z, 2, 'z').copy()
        frame = _f32(rgb_frame, 4, 'RGB')
        if z.shape != (1, 100) or frame.shape != (1, 3, 64, 64):
            raise TypeError("paint_stroke takes z (1,100) and RGB (1,3,64,64)")
        bx = np.array([_int_scalar(v, n) for v, n in zip(box, ('x1', 'y1', 'x2', 'y2'))], np.int32)
        recon = np.ascontiguousarray(recon_u8)
        err = _f32(error, 3, 'error')
        if recon.dtype != np.uint8 or recon.shape != (3, 64, 64) or err.shape != (3, 64, 64):
            raise TypeError("recon_u8 must be uint8 (3,64,64) and error float32 (3,64,64)")
        im = np.empty((3, 64, 64), np.uint8)
        disp = np.empty((256, 256, 3), np.uint8)
        self._check(self._lib.ian_paint_stroke_host(self._h, _fp(z), bx.ctypes.data_as(C.POINTER(C.c_int32)), _fp(frame),
                                                    float(weight), recon.ctypes.data_as(C.c_void_p), _fp(err),
                                                    im.ctypes.data_as(C.c_void_p), disp.ctypes.data_as(C.c_void_p)))
        return z, im, disp

    # ---- multi-GPU: all-gather fused into the decoder's last kernel (peer stores over NVLink) ---------------------
    def setup_fused_gather(self, n_local, group=None):
        """Collective over `group` (torch.distributed, one process per GPU): allocate the gather buffers, exchange
        their CUDA IPC handles and map the peers.  Afterwards reconstruct_gather_dev() decodes straight into every
        rank's buffer: the decoder's last kernel (dec_out for IAN_simple.py, the RGB-Beta head's last kernel for IAN.py
        and IANv1.py) stores each image into every rank's buffer, in the precision set by set_precision().  Needs the
        'tc' path.  Call once per model: the buffers cannot be re-created."""
        import torch
        import torch.distributed as dist
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        mine = (C.c_ubyte * 64)()
        self._check(self._lib.ian_gather_create(self._h, world, rank, int(n_local), C.cast(mine, C.c_void_p)))
        dev = torch.device("cuda", torch.cuda.current_device())
        local = torch.tensor(list(bytes(mine)), dtype=torch.uint8, device=dev)
        allh = torch.empty(world * 64, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(allh, local, group=group)
        blob = bytes(allh.cpu().tolist())
        self._check(self._lib.ian_gather_connect(self._h, C.cast(C.create_string_buffer(blob, len(blob)), C.c_void_p)))
        self._gather_world, self._gather_n = world, int(n_local)

    def reconstruct_gather_dev(self, x_ptr, n_local, z_ptr=0, stream=0):
        """encode -> decode of this rank's shard; returns the device pointer of the (world*n_local,3,64,64) float32
        buffer that holds EVERY rank's decoded images once the stream work (incl. the peer barrier) has run."""
        out = C.c_void_p()
        self._check(self._lib.ian_reconstruct_gather_dev(self._h, x_ptr, int(n_local), z_ptr or None, C.byref(out),
                                                         stream or None))
        return out.value

    def reconstruct_gather_async_dev(self, x_ptr, n_local, z_ptr=0, stream=0):
        """pipelined form: enqueue this rank's shard; a side stream pushes it to the peers (copy engines + stream memory
        operations; IAN_PUSH=kernel: a copy kernel) while the next call computes.  gather_wait_dev() returns the complete buffer of the most recent step."""
        self._check(self._lib.ian_reconstruct_gather_async_dev(self._h, x_ptr, int(n_local), z_ptr or None, stream or None))

    def gather_wait_dev(self, stream=0):
        out = C.c_void_p()
        self._check(self._lib.ian_gather_wait_dev(self._h, C.byref(out), stream or None))
        return out.value

    def reconstruct_sharded(self, x, group=None, stream=0, pipelined=False):
        """Data-parallel encode -> decode of a FULL batch held by every rank (torch CUDA tensor (N,3,64,64) float32, N
        divisible by the world size): this rank computes shard `parallel.shard_bounds(N, rank, world)` and the decoded
        shards are all-gathered by the library (peer stores over NVLink from the decoder's last kernel, or with
        pipelined=True a side-stream push; every graph, either precision).  Returns a torch tensor VIEW (N,3,64,64) of
        the library's gather buffer (valid until the next call's stream work; see include/ian_b200.h)."""
        import torch
        import torch.distributed as dist
        from . import parallel
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        n = int(x.shape[0])
        lo, hi = parallel.shard_bounds(n, rank, world)
        if n % world:
            raise ValueError("reconstruct_sharded needs a batch divisible by the world size (got %d over %d ranks); "
                             "parallel.sharded_reconstruct handles ragged shards with a separate all_gather" % (n, world))
        if getattr(self, '_gather_n', None) != hi - lo or getattr(self, '_gather_world', None) != world:
            if getattr(self, '_gather_n', None) is not None:
                raise _lib.IanError("gather buffers were sized for %d images per rank" % self._gather_n)
            self.setup_fused_gather(hi - lo, group)
        shard = x[lo:hi]
        if pipelined:
            self.reconstruct_gather_async_dev(shard.data_ptr(), hi - lo, 0, stream)
            ptr = self.gather_wait_dev(stream)
        else:
            ptr = self.reconstruct_gather_dev(shard.data_ptr(), hi - lo, 0, stream)
        return parallel.as_cuda_tensor(ptr, (n, 3, 64, 64), x.device)

    # ---- device-pointer variants (ints from torch.Tensor.data_ptr(); no host copies, async) ----------
    def reconstruct_dev(self, x_ptr, n, z_ptr, xhat_ptr, stream=0):
        self._check(self._lib.ian_reconstruct_dev(self._h, x_ptr, n, z_ptr or None, xhat_ptr, stream or None))

    def encode_dev(self, x_ptr, n, z_ptr, eps_ptr=0, stream=0):
        self._check(self._lib.ian_encode_dev(self._h, x_ptr, n, eps_ptr or None, z_ptr, stream or None))

    def decode_dev(self, z_ptr, n, x_ptr, stream=0):
        self._check(self._lib.ian_decode_dev(self._h, z_ptr, n, x_ptr, stream or None))

    def grad_dev(self, z_ptr, boxes_ptr, target_ptr, target_is_frame, n, g_ptr, stream=0):
        self._check(self._lib.ian_grad_dev(self._h, z_ptr, boxes_ptr, target_ptr or None, int(target_is_frame), n,
                                           g_ptr, stream or None))

    def edit_loop_dev(self, z_ptr, boxes_ptr, target_ptr, target_is_frame, n, n_steps, weight, stream=0):
        self._check(self._lib.ian_edit_loop_dev(self._h, z_ptr, boxes_ptr, target_ptr or None, int(target_is_frame),
                                                n, int(n_steps), float(weight), stream or None))
