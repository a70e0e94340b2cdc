"""Generate tests/golden/ref_exec_*.npz by EXECUTING the reference's own Python files.

Theano 0.9 / Lasagne 0.2.dev1 are not installed (and cannot be), so `oracle/refshim/` supplies numpy stand-ins for
those two third-party packages only.  Everything above them is the reference's unmodified code, imported at run time
from its checkout (oracle/reference.py; nothing is copied): `API.IAN.__init__` builds the graph from `IAN_simple.get_model`,
`layers.DeconvLayer` issues its cuDNN calls, `GANcheckpoints.load_weights` loads the checkpoint by parameter name, and
the compiled-function attributes `Z_hat_fn`, `X_hat_fn`, `calculate_lighten_gradient`, `calculate_RGB_gradient` are
the ones `API.py:46-64` defines.  The trained blobs are git-LFS pointers (SURVEY F2), so the checkpoint is the seeded
synthetic one of `oracle/weights.py`, written in the `GANcheckpoints` .npz format next to a symlink of the config
(`API.py:20` derives the weights path from the config path).  Gradients come from the stand-in's `T.grad`, i.e.
central differences of the reference forward in float64.

    python tests/golden/make_golden_ref.py simple        # ~10 min (three numeric gradients)
    python tests/golden/make_golden_ref.py v1 full       # ~6 min with the numeric gradients (REF_EXEC_GRADS=0: ~10 s)

Tests read only the committed .npz files.  The IAN_simple outputs are split over ref_exec_simple.npz and
ref_exec_simple_rand.npz (the decodes of the random latents) so that each file stays under 1 MB.
"""
import json
import logging
import os
import sys
import time

import numpy as np

sys.dont_write_bytecode = True                      # the reference checkout may be read-only
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.reference import reference_dir  # noqa: E402
REF = reference_dir() or sys.exit('no checkout of ajbrock/Neural-Photo-Editor: set NPE_REFERENCE')
sys.path[:0] = [os.path.join(ROOT, 'oracle', 'refshim'), REF]
WORK = os.path.join(ROOT, 'oracle', '_ref', 'work')   # git-ignored scratch: config symlink + synthetic checkpoint
OUT = os.environ.get('REF_EXEC_OUT', os.path.join(ROOT, 'tests', 'golden'))   # the regeneration test writes elsewhere

from oracle import ian_numpy as on      # noqa: E402  (only to_tanh and the weight generator: inputs, not outputs)
from oracle import weights as ow        # noqa: E402


def _stage(config, weights):
    os.makedirs(WORK, exist_ok=True)
    link = os.path.join(WORK, config)
    if os.path.islink(link):
        os.remove(link)
    os.symlink(os.path.join(REF, config), link)
    np.savez(os.path.join(WORK, config[:-3] + '.npz'), **weights)
    return link


def _cfg_json(cfg):
    """the config module's `cfg` dict (API.py:18), JSON with stringified keys"""
    norm = lambda v: {str(k): norm(x) for k, x in v.items()} if isinstance(v, dict) else (list(v) if isinstance(v, tuple) else v)
    return np.array(json.dumps(norm(cfg), sort_keys=True))


def _loader_params(model):
    """the parameter list API.py:24-28 hands to GANcheckpoints.load_weights"""
    import lasagne
    ps = list(set(lasagne.layers.get_all_params(model['l_out'], trainable=True) +
                  lasagne.layers.get_all_params(model['l_discrim'], trainable=True) +
                  [x for x in lasagne.layers.get_all_params(model['l_out']) + lasagne.layers.get_all_params(model['l_discrim'])
                   if x.name[-4:] == 'mean' or x.name[-7:] == 'inv_std']))
    return sorted((p.name, tuple(p.get_value().shape)) for p in ps)


def simple():
    import theano
    import lasagne
    from API import IAN                                   # the reference's API.py
    gold = np.load(os.path.join(ROOT, 'tests', 'golden', 'ian_simple_golden.npz'))   # inputs only: images, z_rand, boxes, rgb
    P = ow.make_simple_weights(int(gold['weight_seed']))
    link = _stage('IAN_simple.py', P)
    out = {}
    for dnn in (True, False):                             # cuDNN DeconvLayer path / plain-Lasagne TransposedConv path
        t0 = time.time()
        m = IAN(config_path=link, dnn=dnn)                # reference API.py:12-64, unmodified
        tag = 'dnn' if dnn else 'nodnn'
        k = 8 if dnn else 2                               # the second wiring only needs to be shown equal: 2 images
        x = on.to_tanh(gold['images'][:k].astype(np.float64)).astype(np.float32)      # NPE.py:257
        z = m.encode_images(x)                            # API.py:78-90
        out['mu_' + tag] = z
        out['xhat_' + tag] = m.sample_at(np.float32(z))   # API.py:98-110 (NPE.py:261 passes float32)
        out['xhat_rand_' + tag] = m.sample_at(gold['z_rand'][:k])
        ls_fn = theano.function([m.X], lasagne.layers.get_output(m.model['l_ls'], {m.model['l_in']: m.X}, deterministic=True))
        out['logsigma_' + tag] = ls_fn(x)
        print(tag, 'forward done in %.1f s' % (time.time() - t0), flush=True)
        if dnn:
            names = _loader_params(m.model)
            out['cfg_json'] = _cfg_json(m.cfg)
            out['model_keys'] = np.array(sorted(m.model.keys()))
            out['param_names'] = np.array([n for n, _ in names])
            out['param_shapes'] = np.array([' '.join(map(str, s)) for _, s in names])
            b = [int(v) for v in gold['boxes'][0]]
            frame = np.broadcast_to(gold['rgb'][0].reshape(1, 3, 1, 1), (1, 3, 64, 64)).astype(np.float32)
            t0 = time.time()
            out['g0_rgb'] = m.imgradRGB(b[0], b[1], b[2], b[3], frame, gold['z_rand'][:2])   # API.py:64,72-76
            out['g0_light'] = m.imgrad(b[0], b[1], b[2], b[3], gold['z_rand'][:2])           # API.py:59,66-70
            b5 = [int(v) for v in gold['boxes'][5]]
            out['g5_box'] = np.array(b5, np.int32)
            frame5 = np.broadcast_to(gold['rgb'][5].reshape(1, 3, 1, 1), (1, 3, 64, 64)).astype(np.float32)
            out['g5_rgb'] = m.imgradRGB(b5[0], b5[1], b5[2], b5[3], frame5, gold['z_rand'][5:6])
            print('numeric gradients done in %.1f s' % (time.time() - t0), flush=True)
    rand = {k: out.pop(k) for k in ('xhat_rand_dnn', 'xhat_rand_nodnn')}
    for name, arrays in (('ref_exec_simple.npz', out), ('ref_exec_simple_rand.npz', rand)):
        path = os.path.join(OUT, name)
        np.savez_compressed(path, **arrays)
        print('wrote', path, os.path.getsize(path), 'bytes')


def flow_model(which):
    """IANv1.py / IAN.py.  The reference's API.IAN cannot construct these (it calls get_model(dnn=...), they define
    get_model(interp=False): SURVEY F6), so the lines of API.IAN.__init__ are followed by hand on the reference's
    own get_model(): parameter list (API.py:24-28), GANcheckpoints.load_weights (:29), MADE reset (:33-36), and the
    compiled functions of API.py:46-51 and sample_IAN.py:84-94."""
    import imp
    import theano
    import theano.tensor as T
    import lasagne
    import GANcheckpoints                                 # the reference's loader
    config = {'v1': 'IANv1.py', 'full': 'IAN.py'}[which]
    gold = np.load(os.path.join(ROOT, 'tests', 'golden', 'ian_%s_golden.npz' % which))   # inputs only
    P = (ow.make_v1_weights if which == 'v1' else ow.make_full_weights)(int(gold['weight_seed']))
    link = _stage(config, P)
    config_module = imp.load_source('config', link)
    model = config_module.get_model()
    params = list(set(lasagne.layers.get_all_params(model['l_out'], trainable=True) +
                      lasagne.layers.get_all_params(model['l_discrim'], trainable=True) +
                      [x for x in lasagne.layers.get_all_params(model['l_out']) + lasagne.layers.get_all_params(model['l_discrim'])
                       if x.name[-4:] == 'mean' or x.name[-7:] == 'inv_std']))
    GANcheckpoints.load_weights(link[:-3] + '.npz', params)
    model['l_IAF_mu'].reset("Once")
    model['l_IAF_ls'].reset("Once")
    X = T.TensorType('float32', [False] * 4)('X')
    Z = T.TensorType('float32', [False] * 2)('Z')
    go = lasagne.layers.get_output
    fns = {
        'Z_hat': theano.function([X], go(model['l_Z'], {model['l_in']: X}, deterministic=True)),          # API.py:50-51
        'X_hat': theano.function([Z], go(model['l_out'], {model['l_Z']: Z}, deterministic=True)),         # API.py:46-47
        'sample': theano.function([Z], go(model['l_out'], {model['l_Z_IAF']: Z}, deterministic=True)),    # sample_IAN.py:84
        'Zfn': theano.function([X], go(model['l_Z_IAF'], {model['l_in']: X}, deterministic=True)),        # sample_IAN.py:89
        'Z_IAF_fn': theano.function([Z], go(model['l_Z'], {model['l_Z_IAF']: Z}, deterministic=True)),    # sample_IAN.py:92
        'logsigma': theano.function([X], go(model['l_ls'], {model['l_in']: X}, deterministic=True)),
    }
    x = on.to_tanh(gold['images'].astype(np.float64)).astype(np.float32)
    names = sorted((p.name, tuple(p.get_value().shape)) for p in params)
    out = {'cfg_json': _cfg_json(config_module.cfg),
           'model_keys': np.array(sorted(model.keys())),
           'param_names': np.array([n for n, _ in names]),
           'param_shapes': np.array([' '.join(map(str, s)) for _, s in names]),
           'ordering_mu': model['l_IAF_mu'].mask_generator.ordering.get_value(),
           'ordering_ls': model['l_IAF_ls'].mask_generator.ordering.get_value(),
           'mask_input': model['l_IAF_mu'].layers[0].weights_mask.get_value(),
           'mask_output_W': model['l_IAF_mu'].layers[1].weights_mask.get_value(),
           'mask_output_D': model['l_IAF_mu'].layers[2].weights_mask.get_value()}
    t0 = time.time()
    out['z'] = fns['Z_hat'](x)
    out['mu'] = fns['Zfn'](x)
    out['logsigma'] = fns['logsigma'](x)
    out['z_from_mu'] = fns['Z_IAF_fn'](np.float32(out['mu']))
    out['xhat'] = fns['X_hat'](np.float32(out['z']))
    out['xhat_rand'] = fns['X_hat'](gold['z_rand'])
    out['sample_rand'] = fns['sample'](gold['z_rand'])
    print(which, 'done in %.1f s' % (time.time() - t0), flush=True)
    if os.environ.get('REF_EXEC_GRADS', '1') != '0':
        # the brush gradients API.py:59,64 would define on this graph (numeric, as for IAN_simple): the target of the
        # next scope row -- the CUDA path has brush gradients for IAN_simple only (DESIGN.md section 8)
        r1, r2 = T.scalar('r1', dtype='int32'), T.scalar('r2', dtype='int32')
        c1, c2 = T.scalar('c', dtype='int32'), T.scalar('c2', dtype='int32')
        RGB = T.tensor4('RGB', dtype='float32')
        X_hat = go(model['l_out'], {model['l_Z']: Z}, deterministic=True)
        lighten = theano.function([c1, r1, c2, r2, Z], T.grad(T.mean(X_hat[0, :, r1:r2, c1:c2]), Z))
        rgbgrad = theano.function([c1, r1, c2, r2, RGB, Z],
                                  T.grad(T.mean((T.sqr(-X_hat[0, :, r1:r2, c1:c2] + RGB[0, :, r1:r2, c1:c2]))), Z))
        box = [20, 24, 33, 37]                                  # c1, r1, c2, r2
        frame = np.broadcast_to(np.float32([0.3, -0.2, 0.6]).reshape(1, 3, 1, 1), (1, 3, 64, 64)).astype(np.float32)
        t0 = time.time()
        out['grad_box'] = np.array(box, np.int32)
        out['grad_rgb_target'] = np.float32([0.3, -0.2, 0.6])
        out['g_light'] = lighten(box[0], box[1], box[2], box[3], gold['z_rand'][:1])
        out['g_rgb'] = rgbgrad(box[0], box[1], box[2], box[3], frame, gold['z_rand'][:1])
        print(which, 'numeric gradients done in %.1f s' % (time.time() - t0), flush=True)
    path = os.path.join(OUT, 'ref_exec_%s.npz' % which)
    np.savez_compressed(path, **out)
    print('wrote', path, os.path.getsize(path), 'bytes')


if __name__ == '__main__':
    import shutil
    logging.basicConfig(level=logging.ERROR)
    try:
        for which in sys.argv[1:] or ['simple', 'v1', 'full']:
            simple() if which == 'simple' else flow_model(which)
    finally:
        shutil.rmtree(WORK, ignore_errors=True)       # 200 MB checkpoints: do not leave them in the tree
