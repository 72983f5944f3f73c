"""Parity of the CUDA path (through the C ABI, via the host mirror `univer_ocr_b200.nn`) with

  1. the golden vectors produced by the unmodified reference (tests/golden/*.npz), and
  2. the float64 oracle (oracle/np_oracle.py) on fresh seeded inputs at larger sizes.

Tolerances (stated per test): the CUDA path stores float32 and accumulates in FP32 FFMA
("check mode", CP.math_mode = fp32); inputs are float32-representable so both sides see the
same numbers.  Max pooling outputs and tie masks, upsampling, window batching and concat are
pure selections/copies and must be BIT-EXACT.
"""
import numpy as np
import pytest

from oracle import np_models, np_oracle as O
from tests.cases import CONV_CASES, MODEL_SHAPES, POOL_CASES

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def nn():
    import univer_ocr_b200.nn as nn_
    nn_.CP.use_gpu()
    nn_.CP.set_math_mode('fp32')
    return nn_


def host(a):
    return np.asarray(a.get() if hasattr(a, 'get') else a, dtype=np.float64)


def close(got, want, rtol=1e-4, atol_scale=2e-6, what=''):
    """|got - want| <= rtol * |want| + atol_scale * max|want| (FP32 accumulate vs float64)."""
    got, want = host(got), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, f'{what}: shape {got.shape} != {want.shape}'
    atol = atol_scale * max(float(np.max(np.abs(want))) if want.size else 0.0, 1e-30)
    np.testing.assert_allclose(got, want, rtol=rtol, atol=atol, err_msg=what)


def f32(a):
    return np.asarray(a, dtype=np.float32).astype(np.float64)


def same_scalar(got, want, rtol):
    """Loss values: NaN must match NaN (the reference's 0 * log 0 SoftmaxCE quirk, losses.py:71)."""
    got, want = float(got), float(want)
    if np.isnan(want) or np.isnan(got):
        return np.isnan(want) and np.isnan(got)
    return abs(got - want) <= rtol * abs(want)


# ----------------------------------------------------------------------------- convolution

@pytest.mark.parametrize('case', CONV_CASES, ids=[c[0] for c in CONV_CASES])
def test_conv2d_golden(nn, golden, case):
    """Convolutional2D fwd / dX / dW / db vs the reference.  rtol 1e-4, atol 2e-6*max."""
    name, _, cin, cout, ks, pad, pv, st = case
    g = golden('conv2d').case(name)
    layer = nn.layers.Convolutional2D(ks, cin, cout, padding=pad, padding_value=pv, stride=st,
                                      w=g['w'], b=g['b'])
    y = layer.forward(g['X'])[0]
    close(y, g['y'], what='y')
    dX = layer.backward(g['dy'])[0]
    close(dX, g['dX'], what='dX')
    close(layer.w.grad, g['dW'], what='dW')
    close(layer.b.grad, g['db'], what='db')


def test_conv2d_grad_accumulates_and_bias_flag(nn, golden):
    """`w.grad += dw` (convolutional.py:138-139) and bias=False (b multiplied by 0, :87,:117)."""
    g = golden('conv2d').case('padval')
    layer = nn.layers.Convolutional2D((4, 4), 6, 7, padding=1, padding_value=0.5, w=g['w'], b=g['b'])
    for _ in range(2):
        layer.forward(g['X'])
        layer.backward(g['dy'])
    close(layer.w.grad, 2 * g['dW'], what='dW x2')
    close(layer.b.grad, 2 * g['db'], what='db x2')
    nob = nn.layers.Convolutional2D((4, 4), 6, 7, padding=1, padding_value=0.5, w=g['w'], b=g['b'],
                                    bias=False)
    close(nob.forward(g['X'])[0], O.conv2d_fwd(g['X'], g['w'], g['b'], 1, 0.5, 1, bias=False), what='y')
    nob.backward(g['dy'])
    assert np.all(host(nob.b.grad) == 0.0)


def test_conv2d_channel_mismatch_raises(nn):
    layer = nn.layers.Convolutional2D((3, 3), 3, 2)
    with pytest.raises(AssertionError):
        layer.forward(np.zeros((1, 5, 5, 4)))


@pytest.mark.parametrize('shape,cin,cout,ks,pad,st', [
    ((3, 62, 92), 1, 16, (3, 3), 1, 1), ((3, 62, 92), 16, 1, (3, 3), 1, 1),
    ((2, 124, 92), 1, 1, (5, 5), 2, 2), ((2, 61, 47), 4, 4, (5, 5), 2, 2),
    ((2, 64, 128), 4, 2, (5, 5), 2, 1), ((3, 32, 70), 1, 64, (5, 3), (0, 1), (2, 1)),
    ((3, 14, 70), 64, 64, (5, 3), (0, 1), (2, 1)), ((2, 33, 35), 5, 3, (4, 2), (2, 1), (3, 2)),
], ids=['mono1', 'mono2', 'para_s2', 'line_s2_odd', 'line_end', 'char1', 'char2', 'odd'])
def test_conv2d_vs_oracle_medium(nn, shape, cin, cout, ks, pad, st):
    """Larger seeded cases against the float64 oracle (rtol 2e-4, atol 4e-6*max)."""
    rng = np.random.default_rng(hash((shape, cin, cout)) % (2 ** 32))
    n, h, w = shape
    X = f32(rng.standard_normal((n, h, w, cin)))
    wt = f32(rng.standard_normal((*ks, cin, cout)) / np.sqrt(ks[0] * ks[1] * cin))
    b = f32(rng.standard_normal(cout))
    layer = nn.layers.Convolutional2D(ks, cin, cout, padding=pad, stride=st, w=wt, b=b)
    y = layer.forward(X)[0]
    want = O.conv2d_fwd(X, wt, b, pad, 0.0, st)
    close(y, want, 2e-4, 4e-6, 'y')
    dy = f32(rng.standard_normal(want.shape))
    dX = layer.backward(dy)[0]
    odX, odW, odb = O.conv2d_bwd(X, wt, dy, pad, 0.0, st)
    close(dX, odX, 2e-4, 4e-6, 'dX')
    close(layer.w.grad, odW, 2e-4, 4e-6, 'dW')
    close(layer.b.grad, odb, 2e-4, 4e-6, 'db')


# ----------------------------------------------------------------------------- pooling etc.

@pytest.mark.parametrize('case', POOL_CASES, ids=[c[0] for c in POOL_CASES])
def test_maxpool_golden_bit_exact(nn, golden, case):
    name, shape, k, pad, st, ceil = case
    g = golden('maxpool2d').case(name)
    layer = nn.layers.MaxPool2D(k, padding=pad, stride=st, ceil_mode=ceil)
    y = layer.forward(g['X'])[0]
    assert np.array_equal(host(y), g['y'])                                   # bit-exact max
    assert np.array_equal(layer._mem[0][0].get(), g['mask'])                 # bit-exact tie mask
    close(layer.backward(g['dy'])[0], g['dX'], 1e-6, 1e-7, 'dX')


def test_maxpool_known_answer(nn, golden):
    g = golden('maxpool2d').case('kat')
    y = nn.layers.MaxPool2D(2, ceil_mode=True).forward(g['X'])[0]
    assert np.array_equal(host(y)[0, :, :, 0], np.array([[1., 2.], [-1., 1.]]))


def test_maxpool_vs_oracle_identity_shape(nn):
    """test_identity.py:81-85 shape family: (5, 240, 320, 6) is scaled to (2, 60, 80, 6)."""
    rng = np.random.default_rng(5)
    X = f32(np.round(rng.standard_normal((2, 60, 80, 6)) * 4) / 4)
    for k, pad, st in ((2, 0, None), (2, 1, None), (2, 0, 1), (2, 1, 1), (3, 1, 2)):
        layer = nn.layers.MaxPool2D(k, padding=pad, stride=st)
        y = layer.forward(X)[0]
        oy, mask = O.maxpool2d_fwd(X, k, pad, st)
        assert np.array_equal(host(y), oy)
        assert np.array_equal(layer._mem[0][0].get(), mask.astype(np.uint8))
        dy = f32(rng.standard_normal(oy.shape))
        close(layer.backward(dy)[0], O.maxpool2d_bwd(dy, mask, X.shape, k, pad, st), 1e-5, 1e-6)


def test_upsample_golden(nn, golden):
    g = golden('upsample2d')
    k = g.case('kat')
    up = nn.layers.Upsample2D((2, 3))
    y = up.forward(k['X'])[0]
    assert np.array_equal(host(y), f32(k['y']))
    close(up.backward(y)[0], k['dX'], 1e-6, 1e-7)
    for name, sf in (('s2', 2), ('s5', 5), ('s23', (2, 3))):
        c = g.case(name)
        up = nn.layers.Upsample2D(sf)
        assert np.array_equal(host(up.forward(c['X'])[0]), c['y'])           # pure copy: exact
        close(up.backward(c['dy'])[0], c['dX'], 1e-6, 1e-6)


def test_elementwise_fc_window_concat_golden(nn, golden):
    g = golden('layers')
    X, dy = g['act__X'], g['act__dy']
    for name, layer in (('relu', nn.layers.Relu()), ('lrelu', nn.layers.LeakyRelu(0.01)),
                        ('lrelu_a', nn.layers.LeakyRelu(0.2)), ('sigmoid', nn.layers.Sigmoid())):
        close(layer.forward(X)[0], g[f'{name}__y'], 2e-6, 1e-7, name)
        close(layer.backward(dy)[0], g[f'{name}__dX'], 2e-6, 1e-7, name)
    fc = nn.layers.FullyConnected(9, 6, w=g['fc__W'])
    close(fc.forward(g['fc__X'])[0], g['fc__y'], 1e-5, 1e-6)
    close(fc.backward(g['fc__dy'])[0], g['fc__dX'], 1e-5, 1e-6)
    close(fc.w.grad, g['fc__dW'], 1e-5, 1e-6)
    for name, width in (('w3', 3), ('w8', 8), ('w8min', 8)):
        c = g.case(f'win_{name}')
        wl = nn.layers.Conv2DToBatchedFixedWidthed(width)
        assert np.array_equal(host(wl.forward(c['X'])[0]), c['y'])            # pure copy: exact
        close(wl.backward(c['dy'])[0], c['dX'], 1e-6, 1e-6)
    cat = nn.layers.Concat()
    y = cat.forward([g['cat__a'], g['cat__b']])[0]
    assert np.array_equal(host(y), g['cat__y'])
    ga, gb = cat.backward([y])
    assert np.array_equal(host(ga), g['cat__ga']) and np.array_equal(host(gb), g['cat__gb'])


def test_fc_vs_oracle_char_head(nn):
    """The three Char FC shapes (513x1024, 1025x128, 129x162) at batch 300."""
    rng = np.random.default_rng(11)
    for n_in, n_out in ((512, 1024), (1024, 128), (128, 162)):
        X = f32(rng.standard_normal((300, n_in)))
        W = f32(rng.uniform(size=(n_in + 1, n_out)) / np.sqrt((n_in + 1) / 2))
        dy = f32(rng.standard_normal((300, n_out)))
        fc = nn.layers.FullyConnected(n_in, n_out, w=W)
        close(fc.forward(X)[0], O.fc_fwd(X, W), 2e-4, 4e-6, 'y')
        odX, odW = O.fc_bwd(X, W, dy)
        close(fc.backward(dy)[0], odX, 2e-4, 4e-6, 'dX')
        close(fc.w.grad, odW, 2e-4, 4e-6, 'dW')


# ----------------------------------------------------------------------------- losses / opt

def test_losses_golden(nn, golden):
    g = golden('losses_opt')
    for name, fn in (('dice', nn.losses.SegmentationDice2D()), ('jaccard', nn.losses.SegmentationJaccard2D())):
        loss, grad = fn(g['seg__pred'], g['seg__gt'])
        assert abs(float(loss) - float(g[f'{name}__loss'])) <= 1e-5 * abs(float(g[f'{name}__loss']))
        close(grad, g[f'{name}__grad'], 1e-5, 1e-6, name)
    loss, grad = nn.losses.SoftmaxCrossEntropy()(g['sce__logits'], g['sce__gt'])
    assert abs(float(loss) - float(g['sce__loss'])) <= 1e-5 * abs(float(g['sce__loss']))
    close(grad, g['sce__grad'], 1e-4, 1e-6)
    loss, grad = nn.losses.SoftmaxCrossEntropy()(g['sce_nan__logits'], g['sce__gt'])
    assert np.isnan(float(loss))                       # 0 * log 0 -> NaN as in the reference
    close(grad, g['sce_nan__grad'], 1e-4, 1e-6)
    loss, grad = nn.losses.SigmoidCrossEntropy()(g['bce__logits'], g['bce__gt'])
    assert abs(float(loss) - float(g['bce__loss'])) <= 1e-5 * abs(float(g['bce__loss']))
    close(grad, g['bce__grad'], 1e-5, 1e-6)


def test_regularisers_and_optimisers_golden(nn, golden):
    g = golden('losses_opt')
    for name, reg in (('l1', nn.regularizations.L1(0.1)), ('l2', nn.regularizations.L2(0.01))):
        loss, grad = reg(g['reg__w'])
        assert abs(float(loss) - float(g[f'{name}__loss'])) <= 1e-6 * abs(float(g[f'{name}__loss']))
        close(grad, g[f'{name}__grad'], 1e-6, 1e-7)
    for name, opt in (('adam', nn.optimizers.Adam(lr=0.0015)),
                      ('momentum', nn.optimizers.Momentum(lr=0.01, momentum=0.9)),
                      ('rmsprop', nn.optimizers.RMSProp(lr=0.01))):
        p = nn.layers.Param(g['reg__w'], optimizer=opt)
        for i, gr in enumerate((g['opt__g1'], g['opt__g2']), start=1):
            p.grad = nn.CP.copy(gr)
            p.update_grad()
            # Adam's first steps are ~3.16*lr*sign(g): compare with an absolute floor (SURVEY 7)
            close(p.value, g[f'{name}__w{i}'], 1e-5, 1e-6, f'{name} step {i}')


def test_dice_large_tile(nn):
    """Dice on a full 496x736 tile: two-pass reduction vs float64 (loss rel 1e-5)."""
    rng = np.random.default_rng(3)
    pred = f32(rng.uniform(0.01, 0.99, size=(2, 496, 736, 1)))
    gt = (rng.uniform(size=pred.shape) < 0.2).astype(np.float64)
    loss, grad = nn.losses.SegmentationDice2D()(pred, gt)
    ol, og = O.dice_loss(pred, gt)
    assert abs(float(loss) - ol) <= 1e-5 * abs(ol)
    close(grad, og, 1e-4, 1e-6)


# ----------------------------------------------------------------------------- whole sub-models

def _check_golden_grads(model, g, step, rtol, atol_frac):
    """Parameter gradients (incl. the L2 term) as the reference had them BEFORE Adam (make_golden.py)."""
    for key, param in model.params().items():
        tag = key.replace('/', '.')
        got = host(param.grad).ravel()
        want = g[f'grad{step}__{tag}__val']
        gmax = float(g[f'grad{step}__{tag}__max'])
        np.testing.assert_allclose(got[g[f'after__{tag}__idx']], want, rtol=rtol, atol=atol_frac * gmax,
                                   err_msg=f'grad{step} {key}')
        l2 = float(np.sqrt((got * got).sum()))
        assert abs(l2 - float(g[f'grad{step}__{tag}__l2'])) <= max(rtol, atol_frac) * float(g[f'grad{step}__{tag}__l2']), key


@pytest.mark.parametrize('fused', [False, True], ids=['per_param', 'fused_update'])
@pytest.mark.parametrize('name', list(MODEL_SHAPES))
def test_submodel_train_golden(nn, golden, name, fused):
    """Two Model.train steps of each my_model sub-network (fwd + loss + bwd + L2 + Adam) vs the reference, on
    un-saturated golden weights (predictions spread over (0, 1): the data gradient is visible next to the L2 term).
    Predictions rtol 1e-4; parameter gradients BEFORE Adam rtol 2e-4 + 5e-6 of the tensor's largest gradient;
    updated weights rtol 1e-3 with an absolute floor of 1e-5 (Adam without bias correction amplifies sign flips of
    near-zero gradients).  `fused`: the steps go through Model.train's flat-buffer update (the default route) instead
    of compute_loss_and_gradients + update_grads + clear_grads; the gradients are then compared on a replica."""
    from univer_ocr_b200 import my_model
    g = golden('models').case(name)
    if name != 'char':
        assert 0.02 < float(g['pred0'].mean()) < 0.98 and float(g['pred0'].std()) > 0.03
    assert float(g['loss1']) != float(g['loss2'])
    w0 = np_models.golden_weights(name, g['seed'])
    opt = nn.optimizers.Adam(lr=0.0015)
    model = my_model.MAKERS[name](MODEL_SHAPES[name], optimizer=opt)
    model.fused_update = fused
    model.set_weights({k: {n: f32(v).tolist() for n, v in p.items()} for k, p in w0.items()})
    close(model.predict(g['X'])[0], g['pred0'], 1e-4, 2e-6, 'pred0')
    for step in (1, 2):
        if fused:
            losses = model.train(g['X'], g['y'])
        else:
            losses = model.compute_loss_and_gradients(g['X'], g['y'])
            # step 2 starts from FP32-updated weights: Adam's ~3.16 lr sign(g) map turns rounding of step-1 gradients
            # that are within 1e-6 of zero into weight differences of ~1e-3, which the step-2 gradients inherit
            _check_golden_grads(model, g, step, 2e-4 if step == 1 else 3e-3, 5e-6 if step == 1 else 1e-4)
            model.update_grads()
            model.clear_grads()
        got = float(losses['output_losses'][0])
        assert abs(got - float(g[f'loss{step}'])) <= 2e-5 * abs(float(g[f'loss{step}'])), (got, g[f'loss{step}'])
        reg = float(losses['regularization_loss'])
        assert abs(reg - float(g[f'reg{step}'])) <= 2e-5 * abs(float(g[f'reg{step}']))
    for key, param in model.params().items():
        tag = f'after__{key.replace("/", ".")}'
        v = host(param.value).ravel()
        np.testing.assert_allclose(v[g[f'{tag}__idx']], g[f'{tag}__val'], rtol=1e-3, atol=1e-5,
                                   err_msg=key)
    close(model.predict(g['X'])[0], g['pred2'], 1e-3, 1e-5, 'pred2')


def test_weights_json_roundtrip(nn, tmp_path):
    """model_weights.json: same keys / nesting as the reference (SURVEY 5), values survive a
    save -> load cycle bit-exactly (float32 -> float64 repr -> float32)."""
    import json
    from univer_ocr_b200 import my_model
    np.random.seed(0)
    models = [my_model.make_monochrome((1, 16, 16, 1)), my_model.make_line((1, 16, 16, 1))]
    path = tmp_path / 'model_weights.json'
    my_model.save_weights(models, path)
    data = json.load(open(path))
    assert set(data) == {'Monochrome/conv_1', 'Monochrome/conv_2', 'Line/down_1/conv_1',
                         'Line/down_2/conv_1', 'Line/up_1/conv_block/conv_1',
                         'Line/up_2/conv_block/conv_1', 'Line/end/conv_1'}
    assert np.array(data['Monochrome/conv_1']['w']).shape == (3, 3, 1, 16)
    assert np.array(data['Line/end/conv_1']['b']).shape == (2,)
    fresh = [my_model.make_monochrome((1, 16, 16, 1)), my_model.make_line((1, 16, 16, 1))]
    my_model.load_weights(fresh, path)
    for a, b in zip(models, fresh):
        for key in a.params():
            assert np.array_equal(a.params()[key].value.get(), b.params()[key].value.get())
    # NaN / shape-mismatch tensors are skipped with a message (layers.py:129-136)
    bad = {'Monochrome/conv_1': {'w': np.full((3, 3, 1, 16), np.nan).tolist(), 'b': [0.0] * 3}}
    before = fresh[0].params()['Monochrome/conv_1/w'].value.get().copy()
    fresh[0].set_weights(bad)
    assert np.array_equal(fresh[0].params()['Monochrome/conv_1/w'].value.get(), before)
    assert not fresh[0].nan_weights()


def test_dag_model_fanout_and_multi_io(nn):
    """Multi-input / multi-output DAG with fan-out (test_gradients.py:225-259 topology), checked
    against the oracle composed by hand: y1 = fc1(flat(pool(cat(c1(x0), c2(x1), c3(x2)))))."""
    rng = np.random.default_rng(21)
    L = nn.layers
    X = [f32(rng.standard_normal((5, 5, 5, 1))) for _ in range(3)]
    ws = [f32(rng.standard_normal((2, 2, 1, 3)) * 0.5) for _ in range(3)]
    bs = [f32(rng.standard_normal(3)) for _ in range(3)]
    W1 = f32(rng.standard_normal((2 * 2 * 9 + 1, 3)) * 0.3)
    W2 = f32(rng.standard_normal((4, 3)) * 0.3)
    layers = {f'conv{i + 1}': L.Convolutional2D((2, 2), out_channels=3, w=ws[i], b=bs[i], in_channels=1)
              for i in range(3)}
    layers.update({'concat': L.Concat(), 'pool': L.MaxPool2D(2), 'flatten': L.Flatten(),
                   'dense1': L.FullyConnected(n_output=3, w=W1, n_input=36),
                   'dense2': L.FullyConnected(n_output=3, w=W2, n_input=3)})
    relations = {'conv1': 0, 'conv2': 1, 'conv3': 2, 'concat': ['conv1', 'conv2', 'conv3'],
                 'pool': 'concat', 'flatten': 'pool', 'dense1': 'flatten', 'dense2': 'dense1',
                 0: 'dense1', 1: 'dense2'}
    model = nn.models.Model(layers, relations, loss=nn.losses.SigmoidCrossEntropy())
    model.initialize_from_X(X)
    y = [(rng.uniform(size=(5, 3)) < 0.5).astype(np.float64) for _ in range(2)]
    out = model.compute_loss_and_gradients(X, y)
    # oracle
    convs = [O.conv2d_fwd(X[i], ws[i], bs[i]) for i in range(3)]
    cat = np.concatenate(convs, axis=-1)
    pooled, mask = O.maxpool2d_fwd(cat, 2)
    flat = pooled.reshape(5, -1)
    d1 = O.fc_fwd(flat, W1)
    d2 = O.fc_fwd(d1, W2)
    l1, g1 = O.sigmoid_ce_loss(d1, y[0])
    l2, g2 = O.sigmoid_ce_loss(d2, y[1])
    assert abs(float(out['output_losses'][0]) - l1) < 1e-5 * abs(l1)
    assert abs(float(out['output_losses'][1]) - l2) < 1e-5 * abs(l2)
    gd1_from2, dW2 = O.fc_bwd(d1, W2, g2)
    gflat, dW1 = O.fc_bwd(flat, W1, g1 + gd1_from2)                 # fan-out: two consumers of dense1
    close(model.layers['dense2'].w.grad, dW2, 1e-4, 2e-6, 'dW2')
    close(model.layers['dense1'].w.grad, dW1, 1e-4, 2e-6, 'dW1')
    gcat = O.maxpool2d_bwd(gflat.reshape(pooled.shape), mask, cat.shape, 2)
    for i in range(3):
        dXi, dWi, _ = O.conv2d_bwd(X[i], ws[i], gcat[..., 3 * i:3 * i + 3])
        close(model.input_grads[i], dXi, 1e-4, 2e-6, f'dX{i}')
        close(model.layers[f'conv{i + 1}'].w.grad, dWi, 1e-4, 2e-6, f'dWconv{i}')


# ----------------------------------------------------------------------------- full-size properties

def test_full_size_adjoint_identities(nn):
    """At BASELINE.json's tile size (496x736; batch 4 here, the identities are batch-independent)
    the oracle is too slow, so check size-independent properties that tie the three conv kernels
    together:  <conv(x) - bias, dy> == <x, dgrad(dy)> == <w, wgrad(x, dy)>  (bilinearity /
    adjointness), and the same adjoint identity for Upsample2D."""
    rng = np.random.default_rng(8)
    for cin, cout, ks, pad, st, hw in ((1, 16, (3, 3), 1, 1, (496, 736)), (16, 1, (3, 3), 1, 1, (496, 736)),
                                       (1, 1, (5, 5), 2, 2, (496, 736)), (4, 4, (5, 5), 2, 1, (128, 256)),
                                       (64, 64, (5, 3), (0, 1), (2, 1), (14, 256))):
        X = f32(rng.standard_normal((4, *hw, cin)))
        wt = f32(rng.standard_normal((*ks, cin, cout)) / np.sqrt(ks[0] * ks[1] * cin))
        layer = nn.layers.Convolutional2D(ks, cin, cout, padding=pad, stride=st, w=wt, b=np.zeros(cout))
        y = host(layer.forward(X)[0])
        dy = f32(rng.standard_normal(y.shape))
        dX = host(layer.backward(dy)[0])
        lhs = float(np.sum(y * dy))
        scale = float(np.sqrt(np.sum(y * y) * np.sum(dy * dy)))
        assert abs(lhs - float(np.sum(X * dX))) <= 2e-5 * scale, (cin, cout, 'dgrad adjoint')
        assert abs(lhs - float(np.sum(wt * host(layer.w.grad)))) <= 2e-5 * scale, (cin, cout, 'wgrad adjoint')
        assert abs(float(np.sum(dy)) - float(np.sum(host(layer.b.grad)))) <= 1e-4 * np.sqrt(dy.size)
    up = nn.layers.Upsample2D(2)
    X = f32(rng.standard_normal((4, 248, 368, 1)))
    y = host(up.forward(X)[0])
    dy = f32(rng.standard_normal(y.shape))
    assert abs(np.sum(y * dy) - np.sum(X * host(up.backward(dy)[0]))) <= 1e-5 * np.sqrt(np.sum(y * y) * np.sum(dy * dy))


def test_row_max_hits_bit_exact(nn):
    """PredToText index rule (interpreter.py:596-602): ties keep all columns, all-zero rows drop."""
    import ctypes
    from univer_ocr_b200._lib import lib
    rng = np.random.default_rng(4)
    pred = f32(np.round(rng.standard_normal((300, 162)) * 2) / 2)
    pred[7, :] = 0.0
    pred[9, :] = -1.0
    d = nn.CP.copy(pred)
    hits = nn.DeviceArray((300, 162), np.uint8)
    lib.uocr_row_max_hits(d.ptr, hits.ptr, 300, 162, nn.CP.stream())
    got = np.argwhere(hits.get() != 0)[:, 1]
    assert np.array_equal(got, O.pred_to_ids(pred))



def test_device_glue_matches_oracle_bit_exact(nn):
    """make_divisible_by / thresholded / pred_to_text on the device (SURVEY.md 8f row 3) are index
    and byte work: bit-exact against the oracle and against the strings recorded from the
    reference's PredToText (tests/golden/glue.json)."""
    import json
    import os
    from univer_ocr_b200 import glue
    rng = np.random.default_rng(21)
    for shape in ((2, 480, 720, 1), (3, 33, 47, 3), (1, 16, 32, 2)):
        a = f32(rng.uniform(size=shape))
        got = host(glue.make_divisible_by(nn.CP.copy(a), 16, 16))
        assert np.array_equal(got, O.make_divisible_by(a, 16, 16))
    for shape in ((4, 496, 736, 1), (5, 128, 256, 2), (3, 7, 5, 8), (1, 1, 1, 1)):
        a = f32(rng.uniform(size=shape) ** 4)                 # skewed like a predicted mask
        a[0] = 0.5                                            # a constant image: empty mask
        mask = glue.thresholded(nn.CP.copy(a)).get()
        assert mask.dtype == np.uint8 and np.array_equal(mask.astype(bool), O.thresholded(a))
        assert not mask[0].any()
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'glue.json')) as fp:
        g = json.load(fp)
    similar = {k: set(v) for k, v in g['similar'].items()}
    for case in g['pred_to_text']:
        text = glue.pred_to_text(nn.CP.copy(np.array(case['pred'])), g['chars'], lambda x, y: x in similar.get(y, ()))
        assert text == case['text']


def test_trainer_epochs_on_device_models(nn):
    """Epoch driver over real networks (SURVEY.md 8f row 1): batches of stacked samples through
    the fused DataParallel step, losses read back once per epoch, device snapshots for the NaN
    roll-back.  The decision logic itself is pinned to the reference in tests/test_trainer.py."""
    from univer_ocr_b200 import my_model
    from univer_ocr_b200.nn.optimizers import Adam
    from univer_ocr_b200.trainer import Trainer
    rng = np.random.default_rng(8)
    opt = Adam(lr=0.002)
    mono = my_model.make_monochrome((1, 32, 48, 1), optimizer=opt)
    char = my_model.make_char((1, 32, 16, 1), optimizer=opt)

    class DS:
        def __init__(self, n, seed):
            r = np.random.default_rng(seed)
            self.items = []
            for _ in range(n):
                x = f32(r.uniform(size=(1, 32, 48, 1)))
                yc = np.zeros((16, 162))
                yc[np.arange(16), r.integers(1, 162, size=16)] = 1
                self.items.append({'mono': (x, f32(x > 0.6)), 'char': (f32(r.uniform(size=(1, 32, 16, 1))), yc)})

        def __len__(self):
            return len(self.items)

        def get(self, i):
            return self.items[i]

    saved, lines = [], []
    trainer = Trainer({'mono': mono, 'char': char}, DS(12, 1), DS(4, 2), optimizer=opt, learning_rate_step=0.9,
                      batch_size=4, save_weights_func=saved.append, log=lambda *a, **k: lines.append(a))
    best, best_epoch = trainer.train(3)
    assert saved and set(saved[-1]) <= {'mono', 'char'}
    assert np.isfinite(best['mono'][0]) and np.isfinite(best['char'][0])
    assert best_epoch['mono'] >= 1
    assert abs(opt.lr - 0.002 * 0.9 ** 3) < 1e-12            # one decay per healthy epoch

    # roll-back path: poison the flat parameter buffer, restore the device snapshot
    st = trainer.steppers['mono']
    X = f32(rng.uniform(size=(2, 32, 48, 1)))
    before = host(mono.predict(X)[0])
    snap = st.snapshot()
    st.train(X, f32(X > 0.5))
    assert np.max(np.abs(host(mono.predict(X)[0]) - before)) > 0
    st.dp.flat.values.fill(float('nan'))
    assert mono.nan_weights()
    st.restore(snap)
    assert not mono.nan_weights()
    assert np.array_equal(host(mono.predict(X)[0]), before)

# ----------------------------------------------------------------------------- fused paths

@pytest.mark.parametrize('name', list(MODEL_SHAPES))
def test_fused_plans_match_unfused(nn, name):
    """Model.fusion (conv+act epilogue, upsample folded into conv, Monochrome conv pair) must give
    the same predictions, losses and gradients as layer-by-layer execution (rtol 1e-5: same FP32
    arithmetic, different association only in the pair kernel)."""
    from univer_ocr_b200 import my_model
    rng = np.random.default_rng(77)
    shape = {'monochrome': (3, 40, 52, 1), 'paragraph': (3, 48, 80, 1), 'line': (3, 32, 48, 1),
             'char': (2, 32, 20, 1)}[name]
    w0 = np_models.golden_weights(name, 99)
    results = []
    for fusion in (False, True):
        nn.models.Model.fusion = fusion
        try:
            model = my_model.MAKERS[name](shape, optimizer=nn.optimizers.Adam(lr=0.002))
        finally:
            nn.models.Model.fusion = True
        model.set_weights({k: {n: v.tolist() for n, v in p.items()} for k, p in w0.items()})
        X = f32(np.random.default_rng(5).uniform(size=shape))
        pred = host(model.predict(X)[0])
        if name == 'char':
            y = np.zeros(pred.shape)
            y[np.arange(y.shape[0]), np.random.default_rng(6).integers(0, y.shape[1], size=y.shape[0])] = 1
        else:
            y = (np.random.default_rng(6).uniform(size=pred.shape) < 0.2).astype(np.float64)
        losses = model.compute_loss_and_gradients(X, y)
        grads = {k: host(p.grad) for k, p in model.params().items()}
        results.append((pred, float(losses['output_losses'][0]), grads, host(model.input_grads[0]),
                        [s[0] for s in model._plan_infer]))
    (p0, l0, g0, dx0, plan0), (p1, l1, g1, dx1, plan1) = results
    assert all(k == 'layer' for k in plan0) and any(k != 'layer' for k in plan1)
    if name == 'monochrome':
        assert plan1 == ['pair']
    close(p1, p0, 1e-5, 1e-6, 'pred')
    assert same_scalar(l1, l0, 1e-5)
    close(dx1, dx0, 1e-4, 1e-6, 'dX')
    for k in g0:
        close(g1[k], g0[k], 1e-4, 2e-6, k)


def test_conv_pair_and_upsample_fusion_edges(nn):
    """Ragged sizes for the fused kernels: widths / heights that are not multiples of the
    per-thread tile (8 columns x 16 rows), 1-pixel images, and odd sizes for upsample+conv."""
    import ctypes
    from univer_ocr_b200._lib import ACT_LEAKY, ACT_SIGMOID, ConvDesc, lib
    rng = np.random.default_rng(31)
    for (n, h, w), c1 in (((2, 1, 1), 16), ((1, 17, 9), 16), ((2, 33, 70), 16), ((1, 16, 64), 5)):
        X = f32(rng.standard_normal((n, h, w, 1)))
        w1 = f32(rng.standard_normal((3, 3, 1, c1)) * 0.4)
        b1 = f32(rng.standard_normal(c1))
        w2 = f32(rng.standard_normal((3, 3, c1, 1)) * 0.3)
        b2 = f32(rng.standard_normal(1))
        hid = O.leaky_relu_fwd(O.conv2d_fwd(X, w1, b1, 1), 0.01)
        want = O.sigmoid_fwd(O.conv2d_fwd(hid, w2, b2, 1))
        d = [nn.CP.copy(a) for a in (X, w1, b1, w2, b2)]
        y = nn.DeviceArray((n, h, w, 1))
        lib.uocr_conv3x3_pair_fwd(d[0].ptr, d[1].ptr, d[2].ptr, d[3].ptr, d[4].ptr, y.ptr, n, h, w, c1,
                                  ACT_LEAKY, 0.01, ACT_SIGMOID, 0.0, 0, nn.CP.stream())
        close(y, want, 1e-4, 2e-6, f'pair {(n, h, w, c1)}')
    for (n, h, w), cin, cout, pad in (((2, 7, 5), 1, 1, 2), ((1, 9, 13), 4, 4, 2), ((2, 6, 11), 4, 2, 2),
                                      ((1, 5, 4), 3, 5, 1)):
        X = f32(rng.standard_normal((n, h, w, cin)))
        wt = f32(rng.standard_normal((5, 5, cin, cout)) * 0.2)
        b = f32(rng.standard_normal(cout))
        want = O.leaky_relu_fwd(O.conv2d_fwd(O.upsample2d_fwd(X, 2), wt, b, pad), 0.01)
        desc = ConvDesc(n, 2 * h, 2 * w, cin, cout, 5, 5, pad, pad, 1, 1, 0.0, 1, 0, 2)
        dx, dw, db = nn.CP.copy(X), nn.CP.copy(wt), nn.CP.copy(b)
        y = nn.DeviceArray(want.shape)
        lib.uocr_conv2d_fwd(ctypes.byref(desc), dx.ptr, dw.ptr, db.ptr, y.ptr, ACT_LEAKY, 0.01,
                            nn.CP.stream())
        close(y, want, 1e-4, 2e-6, f'ups+conv {(n, h, w, cin, cout)}')


@pytest.mark.parametrize('name', list(MODEL_SHAPES))
def test_fused_data_parallel_step_matches_model_train(nn, golden, name):
    """parallel.DataParallel (flat parameter buffers, one fused L2+Adam kernel per group, one
    gradient memset) must reproduce Model.train: same golden losses and updated weights."""
    from univer_ocr_b200 import my_model
    from univer_ocr_b200.parallel import DataParallel
    g = golden('models').case(name)
    w0 = np_models.golden_weights(name, g['seed'])
    opt = nn.optimizers.Adam(lr=0.0015)
    model = my_model.MAKERS[name](MODEL_SHAPES[name], optimizer=opt)
    model.set_weights({k: {n: f32(v).tolist() for n, v in p.items()} for k, p in w0.items()})
    dp = DataParallel(model, optimizer=opt)
    seen = []

    def check_grads():                                    # data gradients before the fused L2 + Adam: golden minus 2*l2*w
        for key, param in model.params().items():
            tag = key.replace('/', '.')
            l2 = 0.01 if '/conv_' in key else 0.0          # my_model/model.py:37-39: L2(0.01) on every conv param
            idx = g[f'after__{tag}__idx']
            want = g[f'grad{len(seen) + 1}__{tag}__val'] - 2 * l2 * host(param.value).ravel()[idx]
            gmax = float(g[f'grad{len(seen) + 1}__{tag}__max'])
            first = not seen
            np.testing.assert_allclose(host(param.grad).ravel()[idx], want, rtol=2e-4 if first else 3e-3,
                                       atol=(5e-6 if first else 1e-4) * gmax, err_msg=key)
        seen.append(1)

    dp.after_reduce = check_grads
    for step in (1, 2):
        losses = dp.train(g['X'], g['y'])
        assert len(seen) == step
        assert same_scalar(losses['output_losses'][0], g[f'loss{step}'], 2e-5)
        assert same_scalar(losses['regularization_loss'], g[f'reg{step}'], 2e-5)
    for key, param in model.params().items():
        tag = f'after__{key.replace("/", ".")}'
        v = host(param.value).ravel()
        np.testing.assert_allclose(v[g[f'{tag}__idx']], g[f'{tag}__val'], rtol=1e-3, atol=1e-5, err_msg=key)
    close(model.predict(g['X'])[0], g['pred2'], 1e-3, 1e-5, 'pred2')


@pytest.mark.parametrize('graph', [False, True], ids=['eager', 'graph'])
def test_inference_pipeline_matches_direct_predict(nn, graph):
    """pipeline.InferencePipeline (three streams, slots, events; per-slot CUDA-graph replay with graph=True) returns,
    in order, exactly what a synchronous predict returns for every submitted batch."""
    from univer_ocr_b200 import my_model
    from univer_ocr_b200.pipeline import InferencePipeline
    np.random.seed(3)
    model = my_model.make_line((4, 32, 64, 1))
    rng = np.random.default_rng(12)
    batches = []
    for _ in range(7):
        buf = nn.CP.pinned_empty((4, 32, 64, 1), np.float32)
        buf[...] = rng.uniform(size=buf.shape)
        batches.append({'x': buf})
    want = [model.predict(np.asarray(b['x']))[0].get() for b in batches]
    pipe = InferencePipeline(lambda inp: model.predict(inp['x']), depth=3, graph=graph)
    got = {}
    for tag, outs in pipe.run(batches):
        got[tag] = outs[0].copy()
    assert sorted(got) == list(range(7))
    for i in range(7):
        assert np.array_equal(got[i], want[i]), i


@pytest.mark.gpu
def test_hourglass_fused_kernel_vs_oracle(nn):
    """uocr_hourglass1_fwd (the whole Paragraph network in one kernel, parity-folded upsample convs)
    vs the float64 oracle chain of five conv layers, for block-aligned, ragged (H, W not multiples of
    the 32 x 128 block), tiny and full-tile sizes, and one grid large enough for the 64-row blocks
    (5 x 512 x 2048: 640 blocks of 64 x 128); FP32 tolerance (rtol 1e-4 + 2e-6 max).
    uocr_hourglass1_fwd_mode runs the same kernel in both math modes: TF32 mode is bit-identical."""
    import ctypes
    from univer_ocr_b200._lib import ACT_NONE, ACT_SIGMOID, MATH_TF32, lib
    rng = np.random.default_rng(123)
    for (n, h, w), act_end in (((2, 32, 128), ACT_SIGMOID), ((1, 36, 140), ACT_NONE), ((3, 4, 4), ACT_SIGMOID),
                               ((2, 8, 300), ACT_NONE), ((1, 132, 12), ACT_SIGMOID), ((1, 496, 736), ACT_SIGMOID),
                               ((2, 496, 736), ACT_SIGMOID), ((1, 64, 2064), ACT_SIGMOID),
                               ((5, 512, 2048), ACT_SIGMOID)):
        X = f32(rng.uniform(size=(n, h, w, 1)))
        ws = [f32(rng.standard_normal((5, 5, 1, 1)) * 0.25) for _ in range(5)]
        bs = [f32(rng.standard_normal(1) * 0.3) for _ in range(5)]
        t = O.leaky_relu_fwd(O.conv2d_fwd(X, ws[0], bs[0], 2, stride=2), 0.01)
        t = O.leaky_relu_fwd(O.conv2d_fwd(t, ws[1], bs[1], 2, stride=2), 0.01)
        t = O.leaky_relu_fwd(O.conv2d_fwd(O.upsample2d_fwd(t, 2), ws[2], bs[2], 2), 0.01)
        t = O.leaky_relu_fwd(O.conv2d_fwd(O.upsample2d_fwd(t, 2), ws[3], bs[3], 2), 0.01)
        want = O.conv2d_fwd(t, ws[4], bs[4], 2)
        if act_end == ACT_SIGMOID:
            want = O.sigmoid_fwd(want)
        dX = nn.CP.copy(X)
        dw = [nn.CP.copy(a) for a in ws]
        db = [nn.CP.copy(a) for a in bs]
        ptrs = ctypes.c_void_p * 5
        y = nn.DeviceArray((n, h, w, 1))
        lib.uocr_hourglass1_fwd(dX.ptr, ptrs(*[a.ptr for a in dw]), ptrs(*[a.ptr for a in db]), y.ptr, n, h, w,
                                0.01, act_end, 0.0, nn.CP.stream())
        close(host(y), want, 1e-4, 2e-6, f'hourglass {(n, h, w)}')
        y_tf32 = nn.DeviceArray.full((n, h, w, 1), -3.0)
        lib.uocr_hourglass1_fwd_mode(dX.ptr, ptrs(*[a.ptr for a in dw]), ptrs(*[a.ptr for a in db]), y_tf32.ptr, n, h,
                                     w, 0.01, act_end, 0.0, MATH_TF32, nn.CP.stream())
        assert np.array_equal(host(y_tf32), host(y)), f'hourglass tf32 mode {(n, h, w)}'


@pytest.mark.gpu
def test_paragraph_predict_uses_hourglass_kernel(nn):
    """Model.predict of make_paragraph takes the fused whole-network kernel (one launch) when H and W
    are multiples of 4, the layer plan otherwise, with the same result either way."""
    from univer_ocr_b200 import my_model
    from univer_ocr_b200._lib import launch_count
    w0 = np_models.golden_weights('paragraph', 99)
    for shape, fused in (((2, 48, 80, 1), True), ((2, 496, 736, 1), True)):
        X = f32(np.random.default_rng(8).uniform(size=shape))
        model = my_model.make_paragraph(shape)
        model.set_weights({k: {n: v.tolist() for n, v in p.items()} for k, p in w0.items()})
        dX = nn.CP.copy(X)
        before = launch_count()
        got = host(model.predict(dX)[0])
        launches = launch_count() - before
        assert (launches == 1) == fused, launches
        hook, model.infer_fusion = model.infer_fusion, None
        ref = host(model.predict(dX)[0])
        model.infer_fusion = hook
        close(got, ref, 1e-4, 2e-6, f'paragraph fused vs layers {shape}')


@pytest.mark.gpu
def test_concurrent_branches_match_serial(nn):
    """pipeline.ConcurrentBranches: the Monochrome -> Paragraph chain, Line and Char forward on three forked CUDA
    streams (own allocator pools) give bit-identical results to the single-stream order, repeatedly (buffers of one
    step are recycled by the next)."""
    from univer_ocr_b200 import my_model
    from univer_ocr_b200.pipeline import ConcurrentBranches
    rng = np.random.default_rng(31)
    shapes = {'monochrome': (2, 64, 96, 1), 'paragraph': (2, 64, 96, 1), 'line': (3, 32, 64, 1), 'char': (2, 32, 40, 1)}
    models = {k: my_model.MAKERS[k](v) for k, v in shapes.items()}
    page = nn.CP.copy(f32(rng.uniform(size=shapes['monochrome'])))
    line = nn.CP.copy(f32(rng.uniform(size=shapes['line'])))
    char = nn.CP.copy(f32(rng.uniform(size=shapes['char'])))
    want = [host(models['paragraph'].predict(models['monochrome'].predict(page)[0])[0]),
            host(models['line'].predict(line)[0]), host(models['char'].predict(char)[0])]
    fork = ConcurrentBranches(3)
    for _ in range(4):
        got = fork.run(lambda: models['paragraph'].predict(models['monochrome'].predict(page)[0])[0],
                       lambda: models['line'].predict(line)[0], lambda: models['char'].predict(char)[0])
        for g, w_ in zip(got, want):
            assert np.array_equal(host(g), w_)


def test_captured_step_replays_match_eager_and_follow_inputs_and_weights(nn):
    """pipeline.CapturedStep: the forked three-stream forward captured into one CUDA graph.  Replays must (a) equal
    the eager result bit for bit, (b) see new data copied into the SAME input buffers, (c) keep working while other
    allocations churn the pool (the graph's blocks are held by the allocator), (d) re-capture after a parameter
    change, and (e) account for the kernels they run in uocr_launch_count."""
    from univer_ocr_b200 import my_model
    from univer_ocr_b200._lib import launch_count
    from univer_ocr_b200.pipeline import CapturedStep, ConcurrentBranches
    rng = np.random.default_rng(32)
    shapes = {'monochrome': (2, 64, 96, 1), 'paragraph': (2, 64, 96, 1), 'line': (3, 32, 64, 1), 'char': (2, 32, 40, 1)}
    models = {k: my_model.MAKERS[k](v) for k, v in shapes.items()}
    for k, m in models.items():                               # signed weights: the default init saturates the sigmoids
        m.set_weights({key: {n: ((v - v.mean()) if n == 'w' else v * 0).tolist() for n, v in p.items()}
                       for key, p in np_models.golden_weights(k, 5).items()})
    host_in = {k: f32(rng.uniform(size=shapes[k])) for k in ('monochrome', 'line', 'char')}
    page, line, char = (nn.CP.copy(host_in[k]) for k in ('monochrome', 'line', 'char'))
    fork = ConcurrentBranches(3)

    def forward():
        return fork.run(lambda: models['paragraph'].predict(models['monochrome'].predict(page)[0])[0],
                        lambda: models['line'].predict(line)[0], lambda: models['char'].predict(char)[0])

    want = [host(o) for o in forward()]
    step = CapturedStep(forward)
    n0 = launch_count()
    got = step()
    per_replay = launch_count() - n0
    assert all(np.array_equal(host(g), w_) for g, w_ in zip(got, want))
    n1 = launch_count()
    step()
    assert launch_count() - n1 >= 10 and launch_count() - n1 <= per_replay     # a replay = the captured kernels
    # (b) + (c): new data in place, allocator churn in between
    page.set(f32(rng.uniform(size=shapes['monochrome'])))
    line.set(f32(rng.uniform(size=shapes['line'])))
    junk = [nn.CP.copy(f32(rng.uniform(size=(64, 64, 7)))) for _ in range(20)]
    del junk
    want2 = [host(o) for o in forward()]
    got2 = step()
    assert all(np.array_equal(host(g), w_) for g, w_ in zip(got2, want2))
    assert not np.array_equal(want2[1], want[1]) and not np.array_equal(want2[0], want[0])
    # (d) parameter change -> re-capture with the new weights
    conv = models['line'].layers['Line/end/conv_1']
    conv.b.value = host(conv.b.value) + 0.5
    want3 = host(forward()[1])
    assert np.array_equal(host(step()[1]), want3) and not np.array_equal(want3, want2[1])
    step.close()


def test_captured_training_step_matches_eager_steps(nn):
    """DataParallel.train captured into a CUDA graph (CapturedStep(track_weights=False)): parameters, gradients and
    Adam state are updated in place, so N replays must leave the same weights and losses as N eager steps
    (tolerance 1e-5 of the largest weight: split-K atomics reorder FP32 sums between any two runs)."""
    from univer_ocr_b200 import my_model
    from univer_ocr_b200.nn.optimizers import Adam
    from univer_ocr_b200.parallel import DataParallel
    from univer_ocr_b200.pipeline import CapturedStep
    rng = np.random.default_rng(41)
    for name, shape in (('line', (3, 32, 64, 1)), ('char', (2, 32, 40, 1))):
        w0 = {key: {n: ((v - v.mean()) if n == 'w' else v * 0).tolist() for n, v in p.items()}
              for key, p in np_models.golden_weights(name, 7).items()}
        X = nn.CP.copy(f32(rng.uniform(size=shape)))
        runs = []
        for mode in ('eager', 'graph'):
            opt = Adam(lr=0.002)
            model = my_model.MAKERS[name](shape, optimizer=opt)
            model.set_weights(w0)
            dp = DataParallel(model, optimizer=opt)
            out_shape = model.get_output_shapes([shape])[0]
            if name == 'char':
                yh = np.zeros(out_shape)
                yh[np.arange(out_shape[0]), np.arange(out_shape[0]) % out_shape[1]] = 1
            else:
                yh = (np.arange(int(np.prod(out_shape))).reshape(out_shape) % 3 == 0).astype(np.float64)
            y = nn.CP.copy(yh)
            dp.train(X, y)                                            # one eager step for both (lazy initialisation)
            step = (lambda: dp.train(X, y)) if mode == 'eager' else CapturedStep(
                lambda: dp.train(X, y), warmup=0, track_weights=False)
            gen0 = nn.CP.weights_generation
            for _ in range(3):
                losses = step()
            runs.append((host(dp.flat.values), float(losses['output_losses'][0]), float(losses['regularization_loss'])))
            if mode == 'graph':
                step.close()
        (we, le, re_), (wg, lg, rg) = runs
        assert np.max(np.abs(we - wg)) <= 1e-5 * np.max(np.abs(we)), name
        assert abs(le - lg) <= 1e-5 * abs(le) and abs(re_ - rg) <= 1e-5 * max(abs(re_), 1e-12), (name, le, lg, re_, rg)


def test_tiled_pooling_and_upsample2_fast_paths_bit_exact(nn):
    """The streaming fast paths (kernel == stride pooling without padding; Upsample2D(2) with C % 4 == 0 or C == 1)
    against the oracle at every vector width, with floor-mode leftover rows / columns, exact ties and odd shapes that
    fall back to the general kernels.  Outputs, tie masks and upsampling are selections: bit-exact; pooling / upsample
    gradients are exact too (one division / three additions in the oracle's order) up to the float32 rounding of it."""
    rng = np.random.default_rng(77)
    for shape, k in (((3, 40, 52, 16), 2), ((2, 31, 29, 6), 3), ((2, 10, 14, 3), 2), ((2, 9, 12, 8), 3), ((1, 7, 5, 4), 2)):
        X = f32(np.round(rng.standard_normal(shape) * 2) / 2)              # many exact ties
        layer = nn.layers.MaxPool2D(k)
        y = layer.forward(X)[0]
        oy, mask = O.maxpool2d_fwd(X, k)
        assert np.array_equal(host(y), oy), (shape, k)
        assert np.array_equal(layer._mem[0][0].get(), mask.astype(np.uint8)), (shape, k)
        dy = f32(rng.standard_normal(oy.shape))
        close(layer.backward(dy)[0], O.maxpool2d_bwd(dy, mask, X.shape, k), 1e-6, 1e-7, f'maxpool dX {shape} k{k}')
    for shape in ((2, 12, 20, 4), (3, 10, 16, 1), (2, 6, 7, 1), (1, 5, 9, 8), (2, 4, 6, 3)):
        X = f32(rng.standard_normal(shape))
        up = nn.layers.Upsample2D(2)
        y = up.forward(X)[0]
        assert np.array_equal(host(y), O.upsample2d_fwd(X, 2)), shape
        dy = f32(rng.standard_normal(host(y).shape))
        close(up.backward(dy)[0], O.upsample2d_bwd(dy, 2), 1e-6, 1e-6, f'upsample dX {shape}')


def test_c_abi_rejects_bad_arguments_with_messages(nn):
    """Error convention of the boundary (include/uocr.h): a negative return code + uocr_last_error() text, nothing
    launched, and the library stays usable afterwards."""
    import ctypes
    from univer_ocr_b200._lib import UocrError, launch_count, lib
    st = nn.CP.stream()
    x = nn.CP.copy(np.ones((1, 4, 4, 1), dtype=np.float32))
    y = nn.DeviceArray((1, 8, 8, 1))
    before = launch_count()
    with pytest.raises(UocrError, match='NULL'):
        lib.uocr_upsample2d_fwd(None, y.ptr, 1, 4, 4, 1, 2, 2, st)
    with pytest.raises(UocrError, match='non-positive'):
        lib.uocr_upsample2d_fwd(x.ptr, y.ptr, 1, 0, 4, 1, 2, 2, st)
    with pytest.raises(UocrError, match='at most 8 channels'):
        work = nn.DeviceArray((1024,), np.uint8)
        lib.uocr_threshold_mask(x.ptr, y.ptr, 1, 1, 16, work.ptr, st)
    with pytest.raises(UocrError, match='kernel larger'):
        ho, wo = ctypes.c_int64(0), ctypes.c_int64(0)
        lib.uocr_maxpool2d_out_hw(2, 2, 3, 3, 0, 0, 1, 1, 0, ctypes.byref(ho), ctypes.byref(wo))
    with pytest.raises(UocrError, match='multiples of 4'):
        ptrs = ctypes.c_void_p * 5
        w5 = [nn.CP.copy(np.zeros((5, 5, 1, 1), dtype=np.float32)) for _ in range(5)]
        b5 = [nn.CP.copy(np.zeros((1,), dtype=np.float32)) for _ in range(5)]
        bad = nn.CP.copy(np.ones((1, 6, 6, 1), dtype=np.float32))
        out = nn.DeviceArray((1, 6, 6, 1))
        lib.uocr_hourglass1_fwd(bad.ptr, ptrs(*[a.ptr for a in w5]), ptrs(*[a.ptr for a in b5]), out.ptr, 1, 6, 6,
                                0.01, 0, 0.0, st)
    assert launch_count() == before                         # nothing was launched by the rejected calls
    lib.uocr_upsample2d_fwd(x.ptr, y.ptr, 1, 4, 4, 1, 2, 2, st)
    assert np.array_equal(y.get(), np.ones((1, 8, 8, 1), dtype=np.float32))


def test_maxpool_full_tile_properties(nn):
    """MaxPool2D(2) / (3) at the microbench's full tile sizes, through properties that need no oracle pass over
    190 M elements: every output equals the maximum of its window and is marked at least once; the gradient of a
    window is shared among its marked positions, so block sums of dX reproduce dy (exactly when a window has one
    winner, to rounding otherwise) and positions outside every window get 0."""
    rng = np.random.default_rng(91)
    for shape, k in (((8, 496, 736, 16), 2), ((16, 240, 320, 6), 3)):
        X = rng.standard_normal(shape).astype(np.float32)
        layer = nn.layers.MaxPool2D(k)
        y = layer.forward(X)[0].get()
        n, h, w, c = shape
        ho, wo = h // k, w // k
        blocks = X[:, :ho * k, :wo * k, :].reshape(n, ho, k, wo, k, c)
        assert np.array_equal(y, blocks.max(axis=(2, 4)))
        mask = layer._mem[0][0].get().reshape(n, ho, k, wo, k, c)
        assert mask.sum(axis=(2, 4)).min() >= 1
        assert np.array_equal(mask.astype(bool), blocks == y[:, :, None, :, None, :])
        dy = rng.standard_normal(y.shape).astype(np.float32)
        dX = layer.backward(dy)[0].get()
        got = dX[:, :ho * k, :wo * k, :].reshape(n, ho, k, wo, k, c).sum(axis=(2, 4), dtype=np.float64)
        assert np.max(np.abs(got - dy)) <= 1e-6 * np.max(np.abs(dy))
        assert not dX[:, ho * k:, :, :].any() and not dX[:, :, wo * k:, :].any()


def test_page_stage_pads_predicts_and_binarises_on_device(nn, tmp_path):
    """predict.PageStage: make_divisible_by -> Monochrome -> Paragraph -> thresholded, weights from model_weights.json,
    against the oracle chain on the same file."""
    from univer_ocr_b200 import weights_io
    from univer_ocr_b200.predict import PageStage
    w = {}
    for name in ('monochrome', 'paragraph'):
        for key, p in np_models.golden_weights(name, 13).items():
            w[key] = {n: ((v - v.mean()) if n == 'w' else v * 0) for n, v in p.items()}    # signed: no saturation
    path = tmp_path / 'model_weights.json'
    weights_io.write(path, w)
    rng = np.random.default_rng(55)
    pages = f32(rng.uniform(size=(2, 100, 150, 1)))
    stage = PageStage(weights_path=path)
    out = stage(pages)
    padded = O.make_divisible_by(pages, 16, 16)
    assert out['padded'].shape == (2, 112, 160, 1) and np.array_equal(host(out['padded']), padded)
    wf = weights_io.read(path)
    mono = np_models.forward(np_models.net_spec('monochrome'), {k: v for k, v in wf.items() if k.startswith('Mono')}, padded)
    para = np_models.forward(np_models.net_spec('paragraph'), {k: v for k, v in wf.items() if k.startswith('Para')}, mono)
    close(out['monochrome_pred'], mono, 1e-4, 1e-5, 'monochrome_pred')
    close(out['paragraph_pred'], para, 1e-4, 1e-5, 'paragraph_pred')
    got = PageStage.to_host(out)
    assert got['paragraph_mask'].dtype == np.uint8 and got['monochrome_pred'].dtype == np.float32
    assert np.array_equal(got['paragraph_mask'].astype(bool), O.thresholded(host(out['paragraph_pred'])))
    assert 0 < got['paragraph_mask'].mean() < 1
    # ... and its connected components, numbered like the reference's label_layer (scipy.ndimage.label of `> mean`)
    from scipy import ndimage
    labels, counts = host(out['paragraph_labels']), host(out['paragraph_count'])
    for i in range(labels.shape[0]):
        layer = got['paragraph_mask'][i:i + 1]
        want, cnt = ndimage.label(layer > np.mean(layer))
        assert cnt == int(counts[i]) and np.array_equal(labels[i:i + 1], want)
    # second call with another page size builds (and caches) another pair of networks
    out2 = stage(f32(rng.uniform(size=(1, 64, 64, 1))))
    assert out2['paragraph_mask'].shape == (1, 80, 80, 1) and len(stage._models) == 2
