"""tests/golden/ref_exec_train.npz: the reference's own MinibatchLayer (layers.py:486-524), executed unmodified from
its checkout (oracle/reference.py) on the numpy stand-ins of oracle/refshim (same mechanism as make_golden_ref.py), plus
the training-mode output of `lasagne.layers.batch_norm` as the reference graphs use it (`BN = batch_norm`,
IAN_simple.py:12) on a conv and a dense layer -- the latter through the stand-in's BatchNormLayer, i.e. restated
third-party semantics.

    python tests/golden/make_golden_train.py
"""
import os
import sys

import numpy as np

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.reference import reference_dir  # noqa: E402
REF = reference_dir() or sys.exit('no checkout of ajbrock/Neural-Photo-Editor: set NPE_REFERENCE')
sys.path[:0] = [os.path.join(ROOT, 'oracle', 'refshim'), REF]
OUT = os.environ.get('REF_EXEC_OUT', os.path.join(ROOT, 'tests', 'golden'))


def main():
    import theano
    import theano.tensor as T
    import lasagne
    import layers as ref_layers                           # the reference's layers.py
    rng = np.random.default_rng(11)
    out = {}
    # ---- MinibatchLayer: n = 6 samples of a (4, 4, 4) feature map (flattened inside, layers.py:504-507), K = 7, P = 5
    n, K, P = 6, 7, 5
    x = rng.standard_normal((n, 4, 4, 4)).astype(np.float32)
    l_in = lasagne.layers.InputLayer((None, 4, 4, 4))
    mb = ref_layers.MinibatchLayer(l_in, num_kernels=K, dim_per_kernel=P, name='minibatch_discrim')
    theta = rng.normal(0, 0.05, (64, K, P)).astype(np.float32)
    lws = rng.normal(0, 0.3, (K, P)).astype(np.float32)
    b = rng.normal(-1, 0.2, (K,)).astype(np.float32)
    mb.theta.set_value(theta); mb.log_weight_scale.set_value(lws); mb.b.set_value(b)
    X = T.TensorType('float32', [False] * 4)('X')
    f = theano.function([X], lasagne.layers.get_output(mb, {l_in: X}))
    out.update(mb_x=x, mb_theta=theta, mb_lws=lws, mb_b=b, mb_out=f(x))
    # ---- batch_norm in training mode (deterministic=False), conv-shaped and dense
    xc = rng.standard_normal((5, 8, 6, 6)).astype(np.float32) * 2 + 0.5
    lc_in = lasagne.layers.InputLayer((None, 8, 6, 6))
    bnc = lasagne.layers.BatchNormLayer(lc_in, name='bn_conv')
    gam = rng.uniform(0.5, 1.5, 8).astype(np.float32); bet = rng.normal(0, 0.1, 8).astype(np.float32)
    bnc.gamma.set_value(gam); bnc.beta.set_value(bet)
    fc = theano.function([X], lasagne.layers.get_output(bnc, {lc_in: X}, deterministic=False))
    out.update(bn_conv_x=xc, bn_conv_gamma=gam, bn_conv_beta=bet, bn_conv_y=fc(xc))
    xd = rng.standard_normal((9, 20)).astype(np.float32) * 3 - 1
    ld_in = lasagne.layers.InputLayer((None, 20))
    bnd = lasagne.layers.BatchNormLayer(ld_in, name='bn_dense')
    gd = rng.uniform(0.5, 1.5, 20).astype(np.float32); bd = rng.normal(0, 0.1, 20).astype(np.float32)
    bnd.gamma.set_value(gd); bnd.beta.set_value(bd)
    X2 = T.TensorType('float32', [False] * 2)('X2')
    fd = theano.function([X2], lasagne.layers.get_output(bnd, {ld_in: X2}, deterministic=False))
    out.update(bn_dense_x=xd, bn_dense_gamma=gd, bn_dense_beta=bd, bn_dense_y=fd(xd))
    path = os.path.join(OUT, 'ref_exec_train.npz')
    np.savez_compressed(path, **out)
    print('wrote', path, os.path.getsize(path), 'bytes')


if __name__ == '__main__':
    main()
