"""Generates tests/golden/*.npz by executing the UNMODIFIED reference (NumPy CPU path) on seeded
inputs.  Needs a checkout of the reference:

    UOCR_REFERENCE_ROOT=<reference checkout> python tests/golden/make_golden.py

The reference has no stored vectors of its own (SURVEY.md 8c); its only fixed cases are the
printed MaxPool / Upsample / Concat examples of nn/test/test_gradients.py:171-188,216-222,
which are reproduced here through the reference's own layers and stored as `kat_*`.
Everything else is the reference run on `numpy.random.default_rng(seed)` inputs.  Inputs are
rounded to float32-representable values so that the CUDA path (float32 storage) and the
float64 reference see *identical* numbers.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import np_models, ref_loader  # noqa: E402
from tests.cases import CONV_CASES, POOL_CASES, MODEL_SHAPES  # noqa: E402


def f32(a):
    return np.asarray(a, dtype=np.float32).astype(np.float64)


def save(name, **arrays):
    path = os.path.join(HERE, name + '.npz')
    np.savez_compressed(path, **arrays)
    print(f'{name}: {os.path.getsize(path) / 1024:.1f} KiB, {len(arrays)} arrays')


def main():
    nn = ref_loader.load_nn()
    L = nn.layers
    rng = np.random.default_rng(20261018)

    # ---------------- convolution ----------------
    out = {}
    for name, (n, h, w), cin, cout, ks, pad, pv, st in CONV_CASES:
        X = f32(rng.standard_normal((n, h, w, cin)))
        wt = f32(rng.standard_normal((*ks, cin, cout)) * 0.3)
        b = f32(rng.standard_normal((cout,)))
        layer = L.Convolutional2D(ks, cin, cout, padding=pad, padding_value=pv, stride=st,
                                  w=wt.copy(), b=b.copy())
        y = layer.forward(X)[0]
        dy = f32(rng.standard_normal(y.shape))
        dX = layer.backward(dy)[0]
        for k, v in dict(X=X, w=wt, b=b, dy=dy, y=y, dX=dX,
                         dW=layer.w.grad, db=layer.b.grad).items():
            out[f'{name}__{k}'] = v
    save('conv2d', **out)

    # ---------------- max pooling ----------------
    out = {}
    for name, shape, k, pad, st, ceil in POOL_CASES:
        # quantised values -> plenty of exact ties, some windows all-negative / all-zero
        X = f32(np.round(rng.standard_normal(shape) * 2) / 2)
        layer = L.MaxPool2D(k, padding=pad, stride=st, ceil_mode=ceil)
        y = layer.forward(X)[0]
        mask = layer._mem[0][0].copy()
        dy = f32(rng.standard_normal(y.shape))
        dX = layer.backward(dy)[0]
        out.update({f'{name}__X': X, f'{name}__dy': dy, f'{name}__y': y,
                    f'{name}__mask': mask.astype(np.uint8), f'{name}__dX': dX})
    # printed known-answer case, test_gradients.py:171-177
    Xk = np.array([[1, 0, 1, 2], [0, -1, -1, -1], [-1, -1, 1, -2]], dtype=np.float64).reshape(1, 3, 4, 1)
    out['kat__X'] = Xk
    out['kat__y'] = L.MaxPool2D(2, ceil_mode=True).forward(Xk)[0]
    save('maxpool2d', **out)

    # ---------------- upsample ----------------
    out = {}
    Xk = np.array([[0.1, 0.2], [0.3, 0.4]]).reshape(1, 2, 2, 1).repeat(4, axis=0).repeat(3, axis=-1)
    up = L.Upsample2D((2, 3))                                     # test_gradients.py:181-188
    yk = up.forward(Xk)[0]
    out.update(kat__X=Xk, kat__y=yk, kat__dX=up.backward(yk)[0])
    for name, shape, sf in (('s2', (2, 5, 7, 4), 2), ('s5', (1, 3, 2, 3), 5), ('s23', (2, 4, 3, 1), (2, 3))):
        X = f32(rng.standard_normal(shape))
        up = L.Upsample2D(sf)
        y = up.forward(X)[0]
        dy = f32(rng.standard_normal(y.shape))
        out.update({f'{name}__X': X, f'{name}__y': y, f'{name}__dy': dy,
                    f'{name}__dX': up.backward(dy)[0]})
    save('upsample2d', **out)

    # ---------------- elementwise layers, FC, window batch, concat ----------------
    out = {}
    X = f32(rng.standard_normal((3, 5, 7, 4)))
    X[0, 0, 0, :2] = 0.0                                          # X == 0 takes the (X >= 0) branch
    dy = f32(rng.standard_normal(X.shape))
    for name, layer in (('relu', L.Relu()), ('lrelu', L.LeakyRelu(0.01)),
                        ('lrelu_a', L.LeakyRelu(0.2)), ('sigmoid', L.Sigmoid())):
        y = layer.forward(X)[0]
        out.update({f'{name}__y': y, f'{name}__dX': layer.backward(dy)[0]})
    out.update(act__X=X, act__dy=dy)
    Xf = f32(rng.standard_normal((5, 9)))
    Wf = f32(rng.standard_normal((10, 6)))
    fc = L.FullyConnected(9, 6, w=Wf.copy())
    yf = fc.forward(Xf)[0]
    dyf = f32(rng.standard_normal(yf.shape))
    out.update(fc__X=Xf, fc__W=Wf, fc__y=yf, fc__dy=dyf, fc__dX=fc.backward(dyf)[0],
               fc__dW=fc.w.grad)
    for name, shape, width in (('w3', (3, 5, 5, 6), 3), ('w8', (2, 1, 11, 64), 8), ('w8min', (1, 2, 8, 3), 8)):
        Xw = f32(rng.standard_normal(shape))
        wl = L.Conv2DToBatchedFixedWidthed(width)
        yw = wl.forward(Xw)[0]
        dyw = f32(rng.standard_normal(yw.shape))
        out.update({f'win_{name}__X': Xw, f'win_{name}__y': yw, f'win_{name}__dy': dyw,
                    f'win_{name}__dX': wl.backward(dyw)[0]})
    cat = L.Concat()                                              # test_gradients.py:216-222
    a, b = np.array([[[1., 2, 3]]]), np.array([[[4., 5, 6]]])
    yc = cat.forward([a, b])[0]
    gc = cat.backward([yc])
    out.update(cat__a=a, cat__b=b, cat__y=yc, cat__ga=gc[0], cat__gb=gc[1])
    save('layers', **out)

    # ---------------- losses, regularisers, optimisers ----------------
    out = {}
    pred = f32(rng.uniform(0.001, 0.999, size=(3, 6, 8, 2)))
    gt = (rng.uniform(size=pred.shape) < 0.3).astype(np.float64)
    gt[2, :, :, 1] = 0.0                                          # an empty-mask channel
    for name, fn in (('dice', nn.losses.SegmentationDice2D()), ('jaccard', nn.losses.SegmentationJaccard2D())):
        loss, grad = fn(pred, gt)
        out.update({f'{name}__loss': np.float64(loss), f'{name}__grad': grad})
    out.update(seg__pred=pred, seg__gt=gt)
    logits = f32(rng.standard_normal((7, 162)) * 3)
    onehot = np.zeros((7, 162))
    onehot[np.arange(7), rng.integers(0, 162, size=7)] = 1
    loss, grad = nn.losses.SoftmaxCrossEntropy()(logits, onehot)
    out.update(sce__logits=logits, sce__gt=onehot, sce__loss=np.float64(loss), sce__grad=grad)
    big = logits.copy()
    big[0, :] = -200.0
    big[0, 3] = 900.0      # p == 0 exactly where gt == 0 -> 0 * log(0) = NaN loss, finite grad
    with np.errstate(all='ignore'):
        loss, grad = nn.losses.SoftmaxCrossEntropy()(big, onehot)
    out.update(sce_nan__logits=big, sce_nan__loss=np.float64(loss), sce_nan__grad=grad)
    bits = (rng.uniform(size=(5, 9)) < 0.5).astype(np.float64)
    lg = f32(rng.standard_normal((5, 9)))
    loss, grad = nn.losses.SigmoidCrossEntropy()(lg, bits)
    out.update(bce__logits=lg, bce__gt=bits, bce__loss=np.float64(loss), bce__grad=grad)
    wv = f32(rng.standard_normal((4, 5)))
    for name, reg in (('l1', nn.regularizations.L1(0.1)), ('l2', nn.regularizations.L2(0.01))):
        loss, grad = reg(wv)
        out.update({f'{name}__loss': np.float64(loss), f'{name}__grad': grad})
    out['reg__w'] = wv
    g1, g2 = f32(rng.standard_normal(wv.shape)), f32(rng.standard_normal(wv.shape) * 1e-3)
    out.update(opt__g1=g1, opt__g2=g2)
    for name, opt in (('adam', nn.optimizers.Adam(lr=0.0015)),
                      ('momentum', nn.optimizers.Momentum(lr=0.01, momentum=0.9)),
                      ('rmsprop', nn.optimizers.RMSProp(lr=0.01))):
        p = L.Param(wv.copy(), optimizer=opt)
        for i, g in enumerate((g1, g2), start=1):
            p.grad = g.copy()
            p.update_grad()
            out[f'{name}__w{i}'] = np.array(p.value)
    save('losses_opt', **out)

    # ---------------- whole sub-models: 2 x Model.train + predict ----------------
    mm = ref_loader.load_my_model()
    shapes = MODEL_SHAPES
    makers = {'monochrome': mm.make_monochrome, 'paragraph': mm.make_paragraph,
              'line': mm.make_line, 'char': mm.make_char}
    out = {}
    for idx, (name, shape) in enumerate(shapes.items()):
        seed = 7000 + idx
        spec = np_models.net_spec(name)
        w0 = np_models.golden_weights(name, seed)
        opt = nn.optimizers.Adam(lr=0.0015)
        model = makers[name](shape, optimizer=opt)
        model.set_weights({k: {n: v.tolist() for n, v in p.items()} for k, p in w0.items()})
        X = f32(rng.uniform(size=shape))
        pred0 = model.predict(X)[0]
        if name == 'char':
            y = np.zeros(pred0.shape)
            y[np.arange(y.shape[0]), rng.integers(0, y.shape[1], size=y.shape[0])] = 1
        else:
            y = (rng.uniform(size=pred0.shape) < 0.2).astype(np.float64)
        if name != 'char':          # the point of golden_weights: predictions spread over (0, 1), not pinned at 1
            assert 0.02 < pred0.mean() < 0.98 and pred0.std() > 0.03, (name, pred0.mean(), pred0.std())
        out.update({f'{name}__seed': np.int64(seed), f'{name}__X': X, f'{name}__y': y,
                    f'{name}__pred0': pred0})
        picks = {}
        for key, param in model.params().items():
            size = int(np.asarray(param.value).size)
            picks[key] = np.random.default_rng(seed + 1).integers(0, size, size=min(size, 96))
        for step in (1, 2):
            # Model.train (nn/models.py:250-254) taken apart so that the gradients can be recorded BEFORE Adam
            # consumes them (they include the L2 term, models.py:246): Adam without bias correction maps any
            # gradient to ~3.16 * lr * sign(g) on the first step, so updated weights alone cannot pin a backward
            losses = model.compute_loss_and_gradients(X, y)
            for key, param in model.params().items():
                g = np.asarray(param.grad, dtype=np.float64).ravel()
                tag = key.replace('/', '.')
                out[f'{name}__grad{step}__{tag}__val'] = g[picks[key]]
                out[f'{name}__grad{step}__{tag}__l2'] = np.float64(np.sqrt((g * g).sum()))
                out[f'{name}__grad{step}__{tag}__max'] = np.float64(np.abs(g).max())
            model.update_grads()
            model.clear_grads()
            out[f'{name}__loss{step}'] = np.float64(losses['output_losses'][0])
            out[f'{name}__reg{step}'] = np.float64(losses['regularization_loss'])
        for key, param in model.params().items():
            v = np.asarray(param.value).ravel()
            pick = picks[key]
            tag = key.replace('/', '.')
            out[f'{name}__after__{tag}__idx'] = pick
            out[f'{name}__after__{tag}__val'] = v[pick]
            out[f'{name}__after__{tag}__sum'] = np.float64(v.sum())
        out[f'{name}__pred2'] = model.predict(X)[0]
    save('models', **out)


if __name__ == '__main__':
    main()
