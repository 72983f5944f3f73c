"""Pins oracle/np_oracle.py + oracle/np_models.py to the reference.

1. Against the committed golden vectors (tests/golden/*.npz, produced by running the
   unmodified reference -- see tests/golden/make_golden.py).  Runs everywhere.
2. Live, against the reference imported from the tree UOCR_REFERENCE_ROOT names, on fresh
   random inputs (`-m reference`-style tests; skipped where that tree is absent).

Tolerance: both sides are float64, only summation order differs -> rtol 1e-10.
"""
import numpy as np
import pytest

from oracle import np_models, np_oracle as O, ref_loader
from tests.cases import CONV_CASES, MODEL_SHAPES, POOL_CASES

RTOL, ATOL = 1e-10, 1e-12


def close(a, b, rtol=RTOL, atol=ATOL):
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol)


@pytest.mark.parametrize('case', CONV_CASES, ids=[c[0] for c in CONV_CASES])
@pytest.mark.parametrize('loop', [False, True], ids=['vec', 'loop'])
def test_conv_golden(golden, case, loop):
    name, _, cin, cout, ks, pad, pv, st = case
    g = golden('conv2d').case(name)
    fwd = O.conv2d_fwd_loop if loop else O.conv2d_fwd
    bwd = O.conv2d_bwd_loop if loop else O.conv2d_bwd
    close(fwd(g['X'], g['w'], g['b'], pad, pv, st), g['y'])
    dX, dW, db = bwd(g['X'], g['w'], g['dy'], pad, pv, st)
    close(dX, g['dX'])
    close(dW, g['dW'])
    close(db, g['db'])


def test_conv_out_shape_and_channel_assert():
    assert O.conv2d_out_hw(13, 11, 5, 2, 2) == (7, 6)
    assert O.conv2d_out_hw(32, 10, (5, 3), (0, 1), (2, 1)) == (14, 10)
    with pytest.raises(AssertionError):
        O.conv2d_fwd(np.zeros((1, 4, 4, 3)), np.zeros((2, 2, 2, 1)), np.zeros(1))


@pytest.mark.parametrize('case', POOL_CASES, ids=[c[0] for c in POOL_CASES])
def test_maxpool_golden(golden, case):
    name, shape, k, pad, st, ceil = case
    g = golden('maxpool2d').case(name)
    y, mask = O.maxpool2d_fwd(g['X'], k, pad, st, ceil)
    assert np.array_equal(y, g['y'])                     # max is exact
    assert np.array_equal(mask.astype(np.uint8), g['mask'])   # tie mask bit-exact
    close(O.maxpool2d_bwd(g['dy'], mask, g['X'].shape, k, pad, st), g['dX'])


def test_maxpool_known_answer(golden):
    """nn/test/test_gradients.py:171-177 prints [[1,2],[-1,1]] for this input."""
    g = golden('maxpool2d').case('kat')
    y, _ = O.maxpool2d_fwd(g['X'], 2, ceil_mode=True)
    assert np.array_equal(y[0, :, :, 0], np.array([[1., 2.], [-1., 1.]]))
    assert np.array_equal(y, g['y'])


def test_upsample_golden(golden):
    g = golden('upsample2d')
    k = g.case('kat')
    y = O.upsample2d_fwd(k['X'], (2, 3))
    assert np.array_equal(y, k['y'])
    close(O.upsample2d_bwd(y, (2, 3)), k['dX'])
    close(O.upsample2d_bwd(y, (2, 3))[0, :, :, 0], np.array([[0.6, 1.2], [1.8, 2.4]]))   # :181-188
    for name, sf in (('s2', 2), ('s5', 5), ('s23', (2, 3))):
        c = g.case(name)
        assert np.array_equal(O.upsample2d_fwd(c['X'], sf), c['y'])
        close(O.upsample2d_bwd(c['dy'], sf), c['dX'])
        close(O.upsample2d_bwd_loop(c['dy'], sf), c['dX'])


def test_elementwise_fc_window_concat_golden(golden):
    g = golden('layers')
    X, dy = g['act__X'], g['act__dy']
    for name, alpha in (('relu', 0.0), ('lrelu', 0.01), ('lrelu_a', 0.2)):
        close(O.leaky_relu_fwd(X, alpha), g[f'{name}__y'])
        close(O.leaky_relu_bwd(X, dy, alpha), g[f'{name}__dX'])
    close(O.sigmoid_fwd(X), g['sigmoid__y'])
    close(O.sigmoid_bwd(X, dy), g['sigmoid__dX'])
    close(O.fc_fwd(g['fc__X'], g['fc__W']), g['fc__y'])
    dX, dW = O.fc_bwd(g['fc__X'], g['fc__W'], g['fc__dy'])
    close(dX, g['fc__dX'])
    close(dW, g['fc__dW'])
    for name, width in (('w3', 3), ('w8', 8), ('w8min', 8)):
        c = g.case(f'win_{name}')
        assert np.array_equal(O.window_batch_fwd(c['X'], width), c['y'])
        close(O.window_batch_bwd(c['dy'], c['X'].shape, width), c['dX'])
    y = O.concat_fwd([g['cat__a'], g['cat__b']])
    assert np.array_equal(y, g['cat__y'])
    ga, gb = O.concat_bwd(y, [g['cat__a'].shape, g['cat__b'].shape])
    assert np.array_equal(ga, g['cat__ga']) and np.array_equal(gb, g['cat__gb'])


def test_losses_regs_optimisers_golden(golden):
    g = golden('losses_opt')
    for name, fn in (('dice', O.dice_loss), ('jaccard', O.jaccard_loss)):
        loss, grad = fn(g['seg__pred'], g['seg__gt'])
        close(loss, g[f'{name}__loss'])
        close(grad, g[f'{name}__grad'])
    loss, grad = O.softmax_ce_loss(g['sce__logits'], g['sce__gt'])
    close(loss, g['sce__loss'])
    close(grad, g['sce__grad'])
    loss, grad = O.softmax_ce_loss(g['sce_nan__logits'], g['sce__gt'])
    assert np.isnan(loss) and np.isnan(g['sce_nan__loss'])          # 0 * log 0, losses.py:71
    close(grad, g['sce_nan__grad'])
    loss, grad = O.sigmoid_ce_loss(g['bce__logits'], g['bce__gt'])
    close(loss, g['bce__loss'])
    close(grad, g['bce__grad'])
    for name, fn, s in (('l1', O.l1_reg, 0.1), ('l2', O.l2_reg, 0.01)):
        loss, grad = fn(g['reg__w'], s)
        close(loss, g[f'{name}__loss'])
        close(grad, g[f'{name}__grad'])
    w, v, a = g['reg__w'], 0.0, 0.0
    for i, gr in enumerate((g['opt__g1'], g['opt__g2']), start=1):
        w, v, a = O.adam_update(w, gr, v, a, lr=0.0015)
        close(w, g[f'adam__w{i}'])
    w, v = g['reg__w'], 0.0
    for i, gr in enumerate((g['opt__g1'], g['opt__g2']), start=1):
        w, v = O.momentum_update(w, gr, v, 0.01, 0.9)
        close(w, g[f'momentum__w{i}'])
    w, a = g['reg__w'], 0.0
    for i, gr in enumerate((g['opt__g1'], g['opt__g2']), start=1):
        w, a = O.rmsprop_update(w, gr, a, 0.01)
        close(w, g[f'rmsprop__w{i}'])


@pytest.mark.parametrize('name', list(MODEL_SHAPES))
def test_submodel_train_golden(golden, name):
    """Two Model.train steps of each my_model sub-network + predict before/after."""
    g = golden('models').case(name)
    spec, kind = np_models.net_spec(name), np_models.loss_kind(name)
    w = np_models.golden_weights(name, g['seed'])
    state = np_models.new_adam_state(w)
    close(np_models.forward(spec, w, g['X']), g['pred0'])
    if name != 'char':                                  # un-saturated: the data gradient is visible next to the L2 term
        assert 0.02 < g['pred0'].mean() < 0.98 and g['pred0'].std() > 0.03
    assert abs(float(g['loss1']) - float(g['loss2'])) > 1e-4 * abs(float(g['loss1']))
    for step in (1, 2):
        losses, grads, _, _ = np_models.train_step(spec, kind, w, state, g['X'], g['y'], lr=0.0015)
        close(losses['output_losses'][0], g[f'loss{step}'], rtol=1e-9)
        close(losses['regularization_loss'], g[f'reg{step}'], rtol=1e-9)
        for key, p in grads.items():                    # gradients (incl. L2) as the reference had them BEFORE Adam
            for n, gr in p.items():
                tag = f'grad{step}__{key}.{n}'.replace('/', '.')
                idx = g[f'after__{key}.{n}__idx'.replace('/', '.')]
                close(gr.ravel()[idx], g[f'{tag}__val'], rtol=1e-8, atol=1e-9 * float(g[f'{tag}__max']))
                close(np.sqrt((gr * gr).sum()), g[f'{tag}__l2'], rtol=1e-8)
    for key, p in w.items():
        for n, v in p.items():
            tag = f'after__{key.replace("/", ".")}/{n}'.replace('/', '.')
            close(v.ravel()[g[f'{tag}__idx']], g[f'{tag}__val'], rtol=1e-8, atol=1e-11)
            close(v.sum(), g[f'{tag}__sum'], rtol=1e-8)
    close(np_models.forward(spec, w, g['X']), g['pred2'], rtol=1e-8)


def test_make_divisible_and_pred_ids():
    a = np.arange(2 * 16 * 30 * 1, dtype=np.float64).reshape(2, 16, 30, 1)
    out = O.make_divisible_by(a, 16, 16)
    assert out.shape == (2, 32, 32, 1)                    # full 16 added when already aligned
    assert np.array_equal(out[:, 8:24, 1:31, :], a)
    pred = np.array([[0.1, 0.7, 0.7], [0.0, 0.0, 0.0], [-1.0, -2.0, -1.5], [0.3, 0.2, 0.1]])
    assert O.pred_to_ids(pred).tolist() == [1, 2, 0, 0]   # ties keep all; all-zero row dropped



def _glue_golden():
    import json
    import os
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'glue.json')) as fp:
        g = json.load(fp)
    similar = {k: set(v) for k, v in g['similar'].items()}
    return g, (lambda a, b: a in similar.get(b, ()))


def test_pred_to_text_and_padding_match_reference_fixture():
    """PredToText._func1 strings and make_divisible_by placements recorded from the reference
    (tests/golden/make_glue_golden.py)."""
    g, are_similar = _glue_golden()
    assert len(g['chars']) == 162
    for case in g['pred_to_text']:
        assert O.pred_to_text(np.array(case['pred']), g['chars'], are_similar) == case['text']
    assert len(g['pred_to_text'][1]['text']) > 64            # tie rows emit several characters
    for pad in g['make_divisible_by']:
        out = O.make_divisible_by(np.ones(pad['shape']), 16, 16)
        ys, xs = np.nonzero(out[0, :, :, 0])
        assert list(out.shape) == pad['out_shape'] and (ys.min(), xs.min()) == (pad['top'], pad['left'])


def test_thresholded_is_mean_max_midpoint_per_image_and_channel():
    rng = np.random.default_rng(3)
    a = rng.uniform(size=(2, 6, 5, 2))
    got = O.thresholded(a)
    for n in range(2):
        for c in range(2):
            sl = a[n, :, :, c:c + 1][None]                   # the (1, H, W, 1) slice the reference passes
            assert np.array_equal(got[n, :, :, c], (sl > 0.5 * (np.mean(sl) + np.max(sl)))[0, :, :, 0])
    assert not O.thresholded(np.ones((1, 4, 4, 1))).any()    # constant map: nothing exceeds its own max

# ------------------------------------------------------------------ live reference diffs

needs_ref = pytest.mark.skipif(not ref_loader.available(), reason='needs the reference tree (UOCR_REFERENCE_ROOT)')


@needs_ref
@pytest.mark.reference
@pytest.mark.parametrize('seed', [1, 2])
def test_live_conv_pool_against_reference(seed):
    """Fresh random inputs through the reference's layers.  Without the reference tree, test_conv_golden and
    test_maxpool_golden check the same oracle functions against what the reference computed."""
    nn = ref_loader.load_nn()
    rng = np.random.default_rng(seed)
    for ks, pad, pv, st in (((3, 3), 1, 0.5, 1), ((5, 5), 2, 0.0, 2), ((5, 3), (0, 1), 0.0, (2, 1)),
                            ((2, 4), (1, 2), -1.0, (3, 1))):
        X = rng.standard_normal((2, 11, 9, 3))
        w = rng.standard_normal((*ks, 3, 4))
        b = rng.standard_normal(4)
        layer = nn.layers.Convolutional2D(ks, 3, 4, padding=pad, padding_value=pv, stride=st,
                                          w=w.copy(), b=b.copy())
        y = layer.forward(X)[0]
        close(O.conv2d_fwd(X, w, b, pad, pv, st), y)
        dy = rng.standard_normal(y.shape)
        dX = layer.backward(dy)[0]
        odX, odW, odb = O.conv2d_bwd(X, w, dy, pad, pv, st)
        close(odX, dX), close(odW, layer.w.grad), close(odb, layer.b.grad)
    for k, pad, st, ceil in ((2, 0, None, False), (3, 1, 2, True), ((2, 3), (1, 1), (1, 2), False)):
        X = np.round(rng.standard_normal((2, 9, 10, 2)) * 2) / 2
        layer = nn.layers.MaxPool2D(k, padding=pad, stride=st, ceil_mode=ceil)
        y = layer.forward(X)[0]
        oy, mask = O.maxpool2d_fwd(X, k, pad, st, ceil)
        assert np.array_equal(oy, y)
        assert np.array_equal(mask, layer._mem[0][0])
        dy = rng.standard_normal(y.shape)
        close(O.maxpool2d_bwd(dy, mask, X.shape, k, pad, st), layer.backward(dy)[0])


@needs_ref
@pytest.mark.reference
def test_live_reference_gradient_suite_subset():
    """The reference's own numeric-gradient check (nn/gradient_check.py) run on its own conv
    layer -- confirms the shimmed reference behaves (full suite: 35/35, SURVEY.md 4)."""
    nn = ref_loader.load_nn()
    rng = np.random.default_rng(0)
    X = rng.standard_normal((2, 5, 5, 3))
    layer = nn.layers.Convolutional2D((3, 3), 3, 2, padding=1, padding_value=0.5, stride=2)
    assert nn.gradient_check.check_layer_gradient(layer, X)
    assert nn.gradient_check.check_layer_param_gradient(layer, X, 'w')


# ---------------------------------------------------------------------------------------------- crop stages (row f4)

def test_stage_resampling_oracle_matches_scipy():
    """oracle/np_stages.py restates SciPy's zoom (order 0) and rotate (order 0 / 1) arithmetic -- pinned against SciPy
    itself on random shapes, zoom factors and angles (incl. the quarter turns and the tie-prone 45 degrees): bit-equal."""
    from scipy import ndimage
    from oracle import np_stages as S
    rng = np.random.default_rng(11)
    for t in range(120):
        h, w, c = int(rng.integers(1, 70)), int(rng.integers(1, 260)), int(rng.integers(1, 3))
        a = rng.uniform(0.1, 1, size=(1, h, w, c)).astype(np.float32)
        zf = int(rng.integers(1, 64)) / h
        want = ndimage.zoom(a, (1, zf, zf, 1), order=0)
        got = S.zoom_nearest(a, zf, zf)
        assert want.shape == got.shape and np.array_equal(want, got), (a.shape, zf)
    for t in range(120):
        h, w, c = int(rng.integers(1, 50)), int(rng.integers(1, 80)), int(rng.integers(1, 3))
        a = rng.uniform(-1, 1, size=(1, h, w, c)).astype(np.float32)
        angle = float(rng.uniform(0, 180)) if t % 4 else float(rng.choice([0, 90, 180, 270, 45, 30, 60, 120, 135]))
        for order in (0, 1):
            want = ndimage.rotate(a, angle, axes=(2, 1), order=order, reshape=True)
            got = S.rotate(a, angle, order)
            assert want.shape == got.shape and np.array_equal(want, got), (a.shape, angle, order)
        m = a[..., :1] > 0
        assert np.array_equal(ndimage.rotate(m, angle, axes=(2, 1), order=0, reshape=True), S.rotate(m, angle, 0))


@needs_ref
def test_stage_oracle_matches_reference_functions():
    """The stage restatements of oracle/np_stages.py against the reference's own functions (interpreter.py:
    label_layer, rearrange_lines, CropRotateAndZoomLines._func1 / _func2, FindObjectHeightInRotated._func,
    rotate_array) on the synthetic cases of tests/stage_cases.py, all four reading directions.  Boolean masks are cast
    to uint8 before the reference's find_objects calls (SciPy 1.18 refuses a boolean maximum label).  Without the
    reference tree, test_stage_oracle_matches_reference_golden checks the line counts, the line crops (zoomed to height 32,
    minimal width 200; they depend on rearrange_lines and line_region), the paragraph angles (the end of the ternary
    search) and the paragraph crops against tests/golden/stages.npz."""
    import importlib
    from scipy import ndimage
    from oracle import np_stages as S
    from tests import stage_cases as C
    ref_loader.load_my_model()
    I = importlib.import_module('web_app.components.interpreter.interpreter')

    def u8(m):
        return m.astype(np.uint8)

    for direction in (None, 90, 180, 270):
        mask, arrays = C.line_paragraph(1, direction)
        top, bottom = S.thresholded(mask[..., 0:1]), S.thresholded(mask[..., 1:2])
        rt, rb, rrot = I.rearrange_lines(I.label_layer(top), I.label_layer(bottom))
        ot, ob, orot = S.rearrange_lines(S.label_layer(top), S.label_layer(bottom))
        assert rrot == orot == direction and len(rt) == len(ot) == 3
        assert all(np.array_equal(a, b) for a, b in zip(rt, ot)) and all(np.array_equal(a, b) for a, b in zip(rb, ob))
        for t, b in zip(rt, rb):
            y, x = I.CropRotateAndZoomLines._func1(u8(t), u8(b))
            assert (y, x) == S.line_region(t, b)
            for arr in arrays:
                for zoomed, minimal in ((32, 200), (32, 1000), (None, 300), (None, None)):
                    want = I.CropRotateAndZoomLines._func2(arr, y, x, rrot, zoomed, minimal)
                    got = S.crop_rotate_zoom(arr, y, x, orot, zoomed, minimal)
                    assert want.shape == got.shape and np.array_equal(want, got)
    pred, images = C.paragraph_page(0)
    res, angles = S.crop_and_rotate_paragraphs(pred, images, True)
    objects = I.label_layer(pred)
    assert len(objects) == len(angles) == 2
    for pid, m in enumerate(objects):
        _, ry, rx, _ = ndimage.find_objects(u8(m))[0]
        cm = u8(m[:, ry, rx, :])
        low, high = 0.0, 180.0
        while high - low > 1.0:                                # CropAndRotateSingleParagraph._func, :318-333
            a, b = low + (high - low) / 3, high - (high - low) / 3
            ha, hb = I.FindObjectHeightInRotated._func(cm, a), I.FindObjectHeightInRotated._func(cm, b)
            assert (ha, hb) == (S.rotated_height(cm, a), S.rotated_height(cm, b))
            if ha < hb:
                high = b
            else:
                low = a
        angle = (high + low) / 2
        assert angle == angles[pid]
        _, oy, ox, _ = ndimage.find_objects(I.rotate_array(cm, angle, good_rotation=False))[0]
        for iid, image in enumerate(images):
            want = I.rotate_array((image * m)[:, ry, rx, :], angle)[:, oy, ox, :]
            assert np.array_equal(want, res[iid][pid])


def test_stage_oracle_matches_reference_golden():
    """oracle/np_stages.py against tests/golden/stages.npz -- outputs of the UNMODIFIED reference's crop-stage functions
    (tests/golden/make_stage_golden.py) on the seeded cases of tests/stage_cases.py: line boxes, zoomed line crops in
    all four reading directions, paragraph angles and straightened paragraph crops, bit for bit."""
    import os
    from oracle import np_stages as S
    from tests import stage_cases as C
    gold = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'stages.npz'))
    for direction in (None, 90, 180, 270):
        mask, arrays = C.line_paragraph(1, direction)
        tag = f'lines_{direction}'
        got = S.crop_rotate_and_zoom_lines([mask], [[a] for a in arrays], 32, 200)
        assert len(got[0][0]) == int(gold[f'{tag}__count']) == 3
        for lid in range(3):
            for aid in range(2):
                assert np.array_equal(got[aid][0][lid], gold[f'{tag}__line{lid}_array{aid}'])
    for seed, tilt in ((0, (12.0, -25.0)), (1, (80.0, 3.0))):
        pred, images = C.paragraph_page(seed, tilt=tilt)
        tag = f'page_{seed}'
        got, angles = S.crop_and_rotate_paragraphs(pred, images, True)
        assert len(angles) == int(gold[f'{tag}__count']) == 2
        for pid in range(2):
            assert angles[pid] == float(gold[f'{tag}__angle{pid}'])
            for iid in range(2):
                assert np.array_equal(got[iid][pid], gold[f'{tag}__par{pid}_image{iid}'])
