"""TF32 tensor-core mode (CP.set_math_mode('tf32')): tcgen05 kernels for FullyConnected and the
Cin % 32 == 0 convolutions against the float64 oracle.

Tolerance (north_star: 1e-3 relative with TF32): |got - want| <= 1e-3 * max|want| elementwise,
and the mean signed relative error on an all-positive problem must be << 1e-3 (TF32 operands are
ROUNDED to nearest by TMA, not truncated by the tensor core, so the error is unbiased).
"""
import os

import numpy as np
import pytest

from oracle import np_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture()
def nn():
    import univer_ocr_b200.nn as nn_
    nn_.CP.use_gpu()
    nn_.CP.set_math_mode('tf32')
    yield nn_
    nn_.CP.set_math_mode('fp32')


def f32(a):
    return np.asarray(a, dtype=np.float32).astype(np.float64)


def close_tf32(got, want, what, tol=1e-3):
    got = np.asarray(got.get() if hasattr(got, 'get') else got, dtype=np.float64)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    err = np.max(np.abs(got - want)) / max(np.max(np.abs(want)), 1e-30)
    assert err <= tol, f'{what}: max err / max|want| = {err:.3e}'
    return err


@pytest.mark.parametrize('batch,n_in,n_out', [(16384, 512, 1024), (1000, 1024, 128), (300, 128, 162),
                                              (129, 36, 20)])
def test_fc_tf32(nn, batch, n_in, n_out):
    rng = np.random.default_rng(batch + n_in)
    X = f32(rng.standard_normal((batch, n_in)))
    W = f32(rng.standard_normal((n_in + 1, n_out)) / np.sqrt(n_in))
    dy = f32(rng.standard_normal((batch, n_out)))
    fc = nn.layers.FullyConnected(n_in, n_out, w=W)
    y = fc.forward(X)[0]
    close_tf32(y, O.fc_fwd(X, W), 'y')
    dX = fc.backward(dy)[0]
    odX, odW = O.fc_bwd(X, W, dy)
    close_tf32(dX, odX, 'dX')
    close_tf32(fc.w.grad, odW, 'dW')


@pytest.mark.parametrize('mode', ['0', '1'])
def test_fc_tf32_cta_pair_kernel(nn, mode, monkeypatch):
    """The persistent GEMM as one CTA per SM (UOCR_TC_PAIR=0) and as CTA pairs sharing 256 x 256 tiles through
    tcgen05 cta_group::2 (=1): same results on a shape with ragged M (tail tile of the second CTA of a pair empty)."""
    monkeypatch.setenv('UOCR_TC_PAIR', mode)
    rng = np.random.default_rng(17)
    batch, n_in, n_out = 16384 + 130, 512, 1024
    X = f32(rng.standard_normal((batch, n_in)))
    W = f32(rng.standard_normal((n_in + 1, n_out)) / np.sqrt(n_in))
    dy = f32(rng.standard_normal((batch, n_out)))
    fc = nn.layers.FullyConnected(n_in, n_out, w=W)
    close_tf32(fc.forward(X)[0], O.fc_fwd(X, W), f'y pair={mode}')
    close_tf32(fc.backward(dy)[0], O.fc_bwd(X, W, dy)[0], f'dX pair={mode}')


def test_fc_tf32_rounding_is_unbiased(nn):
    """All-positive operands: truncation to TF32 would bias every product by ~ -2^-10 and the
    sums by ~ -1e-3 relative; round-to-nearest leaves |mean relative error| below 1e-4."""
    rng = np.random.default_rng(0)
    X = f32(rng.uniform(0.5, 1.5, size=(512, 512)))
    W = f32(rng.uniform(0.5, 1.5, size=(513, 256)))
    fc = nn.layers.FullyConnected(512, 256, w=W)
    y = np.asarray(fc.forward(X)[0].get(), dtype=np.float64)
    want = O.fc_fwd(X, W)
    rel = (y - want) / want
    print('mean signed rel err', rel.mean(), 'max abs rel err', np.abs(rel).max())
    assert abs(rel.mean()) < 1e-4, rel.mean()
    assert np.abs(rel).max() < 1e-3


@pytest.mark.parametrize('shape,cin,cout,ks,pad,st', [
    ((3, 14, 256), 64, 64, (5, 3), (0, 1), (2, 1)),      # Char conv_2
    ((64, 14, 256), 64, 64, (5, 3), (0, 1), (2, 1)),     # Char conv_2 at full batch
    ((3, 5, 256), 64, 64, (5, 3), (0, 1), (2, 1)),       # Char conv_3
    ((2, 14, 70), 64, 64, (5, 3), (0, 1), (2, 1)),       # ragged width (partial 128-pixel tile)
    ((2, 9, 131), 32, 48, (3, 3), (1, 1), (1, 1)),       # other channel counts / square kernel
    ((2, 11, 67), 32, 64, (3, 3), (1, 1), (1, 1)),       # Cin 32: four taps per wgrad CTA
    ((1, 9, 40), 128, 32, (2, 3), (1, 1), (2, 1)),       # Cin 128: one tap per wgrad CTA, even kernel height
], ids=['char2', 'char2_b64', 'char3', 'ragged', 'c32_48', 'c32_64', 'c128_32'])
def test_conv_tf32(nn, shape, cin, cout, ks, pad, st):
    rng = np.random.default_rng(sum(shape) + cin)
    n, h, w = shape
    X = f32(rng.standard_normal((n, h, w, cin)))
    wt = f32(rng.standard_normal((*ks, cin, cout)) / np.sqrt(ks[0] * ks[1] * cin))
    b = f32(rng.standard_normal(cout))
    layer = nn.layers.Convolutional2D(ks, cin, cout, padding=pad, stride=st, w=wt, b=b)
    y = layer.forward(X)[0]
    want = O.conv2d_fwd(X, wt, b, pad, 0.0, st)
    close_tf32(y, want, 'y')
    dy = f32(rng.standard_normal(want.shape))
    dX = layer.backward(dy)[0]
    odX, odW, odb = O.conv2d_bwd(X, wt, dy, pad, 0.0, st)
    close_tf32(dX, odX, 'dX')
    close_tf32(layer.w.grad, odW, 'dW')
    close_tf32(layer.b.grad, odb, 'db')


def test_char_model_tf32_matches_fp32(nn):
    """Whole Char sub-network (inference plan: conv + LeakyRelu epilogues on the tensor-core
    kernels) in TF32 mode vs FP32 check mode: predictions within 2e-3 of max|logit|."""
    from oracle import np_models
    from univer_ocr_b200 import my_model
    shape = (3, 32, 256, 1)
    w0 = np_models.golden_weights('char', 5)
    X = f32(np.random.default_rng(1).uniform(size=shape))
    preds = {}
    for mode in ('fp32', 'tf32'):
        nn.CP.set_math_mode(mode)
        model = my_model.make_char(shape)
        model.set_weights({k: {n: v.tolist() for n, v in p.items()} for k, p in w0.items()})
        preds[mode] = np.asarray(model.predict(X)[0].get(), dtype=np.float64)
    err = np.max(np.abs(preds['tf32'] - preds['fp32'])) / np.max(np.abs(preds['fp32']))
    print('char tf32 vs fp32 max err / max', err)
    assert err < 2e-3


def test_monochrome_pair_on_tensor_cores(nn):
    """uocr_conv3x3_pair_fwd in TF32 mode vs the float64 oracle: |err| <= 1e-3 * max (outputs are sigmoid values in
    (0, 1)) for aligned and ragged sizes (tile / strip / band / step remainders, single-pixel rows and columns,
    odd image counts, several work units per persistent CTA), plus agreement with the FP32 pair kernel.  TF32 mode
    runs csrc/conv_pair_rows_tc.cu (GEMM 1 reads the image rows in shared memory through overlapping descriptor rows)
    where W % 4 == 0 and W >= 8; the other widths (150, 3, 1, 31, 61, 734) take csrc/conv_pair_tc.cu (windows stored to
    tensor memory), 9 x 300 x 734 at several bands per image."""
    import ctypes
    from univer_ocr_b200._lib import ACT_LEAKY, ACT_NONE, ACT_SIGMOID, lib
    rng = np.random.default_rng(17)
    for (n, h, w), act2 in (((2, 16, 256), ACT_SIGMOID), ((3, 21, 150), ACT_SIGMOID), ((1, 5, 3), ACT_NONE),
                            ((2, 1, 1), ACT_NONE), ((1, 63, 31), ACT_SIGMOID), ((1, 130, 61), ACT_NONE),
                            ((5, 3, 240), ACT_SIGMOID), ((2, 496, 736), ACT_SIGMOID), ((3, 33, 244), ACT_SIGMOID),
                            ((2, 40, 248), ACT_NONE), ((1, 7, 492), ACT_SIGMOID), ((1, 130, 1000), ACT_SIGMOID),
                            ((5, 3, 12), ACT_NONE), ((1, 2, 8), ACT_SIGMOID), ((9, 300, 736), ACT_SIGMOID),
                            ((9, 300, 734), ACT_NONE)):
        X = f32(rng.uniform(size=(n, h, w, 1)))
        w1 = f32(rng.standard_normal((3, 3, 1, 16)) * 0.4)
        b1 = f32(rng.standard_normal(16) * 0.2)
        w2 = f32(rng.standard_normal((3, 3, 16, 1)) * 0.3)
        b2 = f32(rng.standard_normal(1))
        hid = O.leaky_relu_fwd(O.conv2d_fwd(X, w1, b1, 1), 0.01)
        want = O.conv2d_fwd(hid, w2, b2, 1)
        if act2 == ACT_SIGMOID:
            want = O.sigmoid_fwd(want)
        d = [nn.CP.copy(a) for a in (X, w1, b1, w2, b2)]
        outs = {}
        # math mode 0 = FP32 pair kernel, 1 = tensor cores; the capped grids put many work units on each CTA
        for key, mode, grid in (('fp32', 0, None), ('tf32', 1, None), ('tf32_1cta', 1, '1'), ('tf32_5cta', 1, '5')):
            if grid is not None and n * h * w > 2000000:
                continue                                # the capped-grid runs exist for the multi-unit bookkeeping
            if grid is not None:
                os.environ['UOCR_PAIR_ROWS_GRID'] = grid      # few persistent CTAs: many work units per CTA
            try:
                y = nn.DeviceArray((n, h, w, 1))
                lib.uocr_conv3x3_pair_fwd(d[0].ptr, d[1].ptr, d[2].ptr, d[3].ptr, d[4].ptr, y.ptr, n, h, w, 16,
                                          ACT_LEAKY, 0.01, act2, 0.0, mode, nn.CP.stream())
                outs[key] = np.asarray(y.get(), dtype=np.float64)
            finally:
                os.environ.pop('UOCR_PAIR_ROWS_GRID', None)
        for key in outs:
            if key == 'fp32':
                continue
            close_tf32(outs[key], want, f'{key} pair {(n, h, w)}')
            close_tf32(outs[key], outs['fp32'], f'{key} vs fp32 pair {(n, h, w)}')


@pytest.mark.parametrize('shape,cout,ups', [
    ((2, 128, 256), 4, 1), ((2, 128, 256), 2, 1),          # Line up_1 (after its upsample) / end
    ((2, 64, 128), 4, 2), ((3, 32, 64), 4, 2),             # Line up_1 / up_2 reading through the folded upsample
    ((1, 37, 45), 4, 1), ((2, 5, 3), 2, 1), ((1, 30, 70), 2, 2), ((1, 1, 1), 4, 1),   # ragged strips / bands
], ids=['up1', 'end', 'up1_ups', 'up2_ups', 'ragged4', 'tiny2', 'ragged_ups', 'one_px'])
def test_conv55_row_gemm_tf32(nn, shape, cout, ups):
    """5x5 / stride 1 / Cin = 4 convolutions as a tcgen05 row GEMM with TMEM-resident windows
    (csrc/conv_row_tc.cu), plain and through a folded Upsample2D(2), + LeakyRelu / Sigmoid epilogue,
    vs the float64 oracle at the TF32 tolerance."""
    import ctypes
    from univer_ocr_b200._lib import ACT_LEAKY, ACT_SIGMOID, ConvDesc, MATH_TF32, lib
    rng = np.random.default_rng(sum(shape) + cout + ups)
    n, h, w = shape                                          # stored input size
    X = f32(rng.standard_normal((n, h, w, 4)))
    wt = f32(rng.standard_normal((5, 5, 4, cout)) / 10.0)
    b = f32(rng.standard_normal(cout) * 0.3)
    Xin = O.upsample2d_fwd(X, 2) if ups == 2 else X
    want = O.conv2d_fwd(Xin, wt, b, 2, 0.0, 1)
    for act, fn in ((ACT_LEAKY, lambda t: O.leaky_relu_fwd(t, 0.01)), (ACT_SIGMOID, O.sigmoid_fwd)):
        desc = ConvDesc(n, h * ups, w * ups, 4, cout, 5, 5, 2, 2, 1, 1, 0.0, 1, MATH_TF32, ups)
        dX, dw, db = nn.CP.copy(X), nn.CP.copy(wt), nn.CP.copy(b)
        y = nn.DeviceArray((n, h * ups, w * ups, cout))
        before = ctypes.c_uint64(0)
        lib.uocr_conv2d_fwd(ctypes.byref(desc), dX.ptr, dw.ptr, db.ptr, y.ptr, act, 0.01, nn.CP.stream())
        close_tf32(y, fn(want), f'row gemm {shape} cout {cout} ups {ups} act {act}')


def test_kmajor_weight_cache_follows_updates(nn):
    """Inference in TF32 mode caches K-major weight copies per layer (uocr_*_fwd_kmajor).  The cache must be
    dropped by every way parameters change: Model.train (optimizer update), DataParallel's flat-buffer update and
    set_weights -- checked against the FP32 mode (which has no cache) of the same model after each change."""
    from oracle import np_models
    from univer_ocr_b200 import my_model
    from univer_ocr_b200.parallel import DataParallel
    rng = np.random.default_rng(3)
    shape = (2, 32, 256, 1)
    w0 = np_models.golden_weights('char', 5)
    opt = nn.optimizers.Adam(lr=0.05)                      # large steps: a stale cache is unmistakable
    model = my_model.make_char(shape, optimizer=opt)
    model.set_weights({k: {n: v.tolist() for n, v in p.items()} for k, p in w0.items()})
    X = f32(rng.uniform(size=shape))
    y = np.zeros((shape[0] * shape[2], 162))
    y[np.arange(y.shape[0]), rng.integers(0, 162, size=y.shape[0])] = 1

    def check(what, prev=None):
        nn.CP.set_math_mode('tf32')
        got = np.asarray(model.predict(X)[0].get(), dtype=np.float64)
        nn.CP.set_math_mode('fp32')
        want = np.asarray(model.predict(X)[0].get(), dtype=np.float64)
        nn.CP.set_math_mode('tf32')
        close_tf32(got, want, what, tol=3e-3)
        if prev is not None:
            assert np.max(np.abs(got - prev)) > 1e-2 * np.max(np.abs(prev)), f'{what}: predictions did not move'
        return got

    p0 = check('initial')
    model.train(X, y)
    p1 = check('after Model.train', p0)
    dp = DataParallel(model, optimizer=opt)
    dp.train(nn.CP.copy(X), nn.CP.copy(y))
    p2 = check('after DataParallel.train', p1)
    w1 = np_models.golden_weights('char', 6)
    model.set_weights({k: {n: v.tolist() for n, v in p.items()} for k, p in w1.items()})
    check('after set_weights', p2)


@pytest.mark.parametrize('n,w,c,width,n_out', [(64, 256, 64, 8, 1024), (48, 128, 32, 8, 256), (3, 200, 64, 8, 1024),
                                              (2, 256, 48, 6, 200)],
                         ids=['char_head', 'small', 'w_not_128', 'c_not_32'])
def test_window_fc_fused(nn, n, w, c, width, n_out):
    """uocr_window_fc_fwd: Conv2DToBatchedFixedWidthed + Flatten + FullyConnected (+ LeakyRelu) in one call -- with the
    window matrix gathered by TMA inside the persistent tcgen05 GEMM (first two cases), or through scratch (other
    geometries) -- vs the float64 oracle of the three layers."""
    from univer_ocr_b200._lib import ACT_LEAKY, MATH_TF32, lib
    rng = np.random.default_rng(n + w + c)
    X = f32(rng.standard_normal((n, 1, w, c)))
    W = f32(rng.standard_normal((width * c + 1, n_out)) / np.sqrt(width * c))
    win = O.window_batch_fwd(X, width)
    want = O.leaky_relu_fwd(O.fc_fwd(win.reshape(n * w, -1), W), 0.01)
    dX, dW = nn.CP.copy(X), nn.CP.copy(W)
    for cached in (False, True):
        wt = None
        if cached:
            wt = nn.DeviceArray((n_out, width * c))
            lib.uocr_weights_to_kmajor(dW.ptr, wt.ptr, width * c, n_out, nn.CP.stream())
        y = nn.DeviceArray((n * w, n_out))
        lib.uocr_window_fc_fwd(dX.ptr, dW.ptr, wt.ptr if wt is not None else None, y.ptr, n, w, c, width, n_out,
                               ACT_LEAKY, 0.01, MATH_TF32, nn.CP.stream())
        close_tf32(y, want, f'window fc {(n, w, c, width, n_out)} cached={cached}')


def test_line_conv_backward_tf32(nn):
    """5x5 4 -> 4 convolution (Line up_*) in TF32 mode: forward and the input gradient both run on the tcgen05 row-GEMM
    kernel (the dgrad as a bias-less forward on flipped weights), the weight gradient on the FP32 stencil; vs oracle."""
    rng = np.random.default_rng(11)
    X = f32(rng.standard_normal((2, 37, 70, 4)))
    wt = f32(rng.standard_normal((5, 5, 4, 4)) / 10.0)
    b = f32(rng.standard_normal(4) * 0.3)
    layer = nn.layers.Convolutional2D((5, 5), 4, 4, padding=2, w=wt, b=b)
    y = layer.forward(X)[0]
    want = O.conv2d_fwd(X, wt, b, 2, 0.0, 1)
    close_tf32(y, want, 'y')
    dy = f32(rng.standard_normal(want.shape))
    dX = layer.backward(dy)[0]
    odX, odW, odb = O.conv2d_bwd(X, wt, dy, 2, 0.0, 1)
    close_tf32(dX, odX, 'dX')
    close_tf32(layer.w.grad, odW, 'dW')
    close_tf32(layer.b.grad, odb, 'db')


def test_full_page_monochrome_paragraph_tf32(nn):
    """BASELINE configs[3] geometry: one 2048 x 2048 document -> make_divisible_by -> (1, 2064, 2064, 1) through
    Monochrome -> Paragraph with the fused tcgen05 / whole-network kernels (TF32 mode) vs the layer-by-layer FP32
    check mode (Model.fusion off): sigmoid outputs within 2e-3."""
    from oracle import np_models
    from univer_ocr_b200 import my_model
    rng = np.random.default_rng(21)
    page = my_model.make_divisible_by(f32(rng.uniform(size=(1, 2048, 2048, 1))), 16, 16)
    assert page.shape == (1, 2064, 2064, 1)
    outs = {}
    for mode, fusion in (('fp32', False), ('tf32', True)):
        nn.CP.set_math_mode(mode)
        nn.models.Model.fusion = fusion
        try:
            mono = my_model.make_monochrome(page.shape)
            para = my_model.make_paragraph(page.shape)
        finally:
            nn.models.Model.fusion = True
        for name, model in (('monochrome', mono), ('paragraph', para)):
            w0 = np_models.golden_weights(name, 99)
            model.set_weights({k: {n: v.tolist() for n, v in p.items()} for k, p in w0.items()})
        m = mono.predict(page)[0]
        outs[mode] = (np.asarray(m.get(), dtype=np.float64), np.asarray(para.predict(m)[0].get(), dtype=np.float64))
    nn.CP.set_math_mode('tf32')
    for i, what in enumerate(('monochrome', 'paragraph')):
        err = np.max(np.abs(outs['tf32'][i] - outs['fp32'][i]))
        # sigmoid outputs in (0, 1).  Monochrome: one TF32 layer pair.  Paragraph reads that map through five more
        # layers whose (un-saturated, centred) weights amplify the input error before the last sigmoid: 4e-3
        assert err <= (2e-3 if what == 'monochrome' else 4e-3), (what, err)


def test_monochrome_pair_backward_tensor_core(nn):
    """uocr_conv3x3_pair_bwd_mode in TF32 mode (hidden map and its gradient recomputed by one tcgen05 GEMM per 128
    pixels, pixel sums on the CUDA cores; csrc/conv_pair_bwd_tc.cu) vs the FP32 CUDA-core kernel and, on the small
    cases, the float64 oracle: dw1, db1, dw2, db2 within 1e-3 of their range; ragged strips / bands / steps.

    LeakyReLU's derivative jumps at h = 0, so an element whose h is below the TF32 resolution can legitimately fall on
    either side.  Two modes are checked: (a) UOCR_PAIR_WGRAD_EXACT_MASK=1 -- borderline h recomputed in FP32 -- on data
    that crosses the kink (random weights, many h near 0) must match the FP32 kernel; (b) the default (branch taken on
    the TF32 h) on data whose h stays away from 0 (|b1| dominates) must match as well."""
    import ctypes
    from univer_ocr_b200._lib import ACT_LEAKY, ACT_NONE, lib
    rng = np.random.default_rng(29)
    for exact in (True, False):
        for (n, h, w), act1 in (((2, 16, 256), ACT_LEAKY), ((3, 21, 150), ACT_LEAKY), ((1, 5, 3), ACT_NONE),
                                ((2, 1, 1), ACT_LEAKY), ((1, 130, 61), ACT_LEAKY), ((2, 496, 736), ACT_LEAKY)):
            X = f32(rng.uniform(size=(n, h, w, 1)))
            if exact:
                w1 = f32(rng.standard_normal((3, 3, 1, 16)) * 0.4)
                b1 = f32(rng.standard_normal(16) * 0.2)
            else:                                   # |h| >= 1.5 - 9 * 0.15: never near the kink, both signs present
                w1 = f32(rng.uniform(-0.15, 0.15, size=(3, 3, 1, 16)))
                b1 = f32(np.where(np.arange(16) % 2 == 0, 1.5, -1.5) + rng.uniform(-0.1, 0.1, size=16))
            w2 = f32(rng.standard_normal((3, 3, 16, 1)) * 0.3)
            dy = f32(rng.standard_normal((n, h, w, 1)))
            d = [nn.CP.copy(a) for a in (X, w1, b1, w2, dy)]
            need = ctypes.c_size_t(0)
            lib.uocr_conv3x3_pair_bwd_workspace(n, h, w, 16, ctypes.byref(need))
            outs = []
            os.environ['UOCR_PAIR_WGRAD_EXACT_MASK'] = '1' if exact else '0'
            try:
                for mode in (0, 1):
                    ws = nn.DeviceArray(((need.value + 3) // 4,))
                    g = [nn.DeviceArray.zeros(s_) for s_ in ((3, 3, 1, 16), (16,), (3, 3, 16, 1), (1,), (n, h, w, 1))]
                    lib.uocr_conv3x3_pair_bwd_mode(d[0].ptr, d[1].ptr, d[2].ptr, d[3].ptr, d[4].ptr, g[4].ptr, g[0].ptr,
                                                   g[1].ptr, g[2].ptr, g[3].ptr, n, h, w, 16, act1, 0.01, 0, ws.ptr,
                                                   need.value, mode, nn.CP.stream())
                    outs.append([np.asarray(t.get(), dtype=np.float64) for t in g])
            finally:
                os.environ.pop('UOCR_PAIR_WGRAD_EXACT_MASK', None)
            # sums over a handful of pixels have no averaging of the per-product TF32 rounding: 2e-3 there
            tol = 2e-3 if n * h * w < 64 else 1e-3
            # dx (conv3x3_pair_dgrad in the TF32 dispatch) is checked too: round 1 passed dx = NULL here
            for name, a, b in zip(('dw1', 'db1', 'dw2', 'db2', 'dx'), outs[1], outs[0]):
                close_tf32(a, b, f'pair bwd tc vs fp32 {name} {(n, h, w)} exact={exact}', tol=tol)
            if h * w <= 4000:
                hid = O.conv2d_fwd(X, w1, b1, 1)
                act = O.leaky_relu_fwd(hid, 0.01) if act1 == ACT_LEAKY else hid
                dact, odw2, odb2 = O.conv2d_bwd(act, w2, dy, 1, 0.0, 1)
                dhid = dact * np.where(hid >= 0, 1.0, 0.01) if act1 == ACT_LEAKY else dact
                odx, odw1, odb1 = O.conv2d_bwd(X, w1, dhid, 1, 0.0, 1)
                for name, a, b in zip(('dw1', 'db1', 'dw2', 'db2', 'dx'), outs[1], (odw1, odb1, odw2, odb2, odx)):
                    close_tf32(a, np.asarray(b, dtype=np.float64).reshape(a.shape),
                               f'pair bwd tc vs oracle {name} {(n, h, w)} exact={exact}', tol=tol)


def _line_oracle(X, ws, bs, act_end, alpha=0.01, alpha_end=0.0):
    """make_line's forward (my_model/model.py:194-248) from the oracle's layers."""
    from univer_ocr_b200._lib import ACT_LEAKY, ACT_SIGMOID
    t = O.leaky_relu_fwd(O.conv2d_fwd(X, ws[0], bs[0], 2, stride=2), alpha)
    t = O.leaky_relu_fwd(O.conv2d_fwd(t, ws[1], bs[1], 2, stride=2), alpha)
    t = O.leaky_relu_fwd(O.conv2d_fwd(O.upsample2d_fwd(t, 2), ws[2], bs[2], 2), alpha)
    t = O.leaky_relu_fwd(O.conv2d_fwd(O.upsample2d_fwd(t, 2), ws[3], bs[3], 2), alpha)
    want = O.conv2d_fwd(t, ws[4], bs[4], 2)
    if act_end == ACT_SIGMOID:
        want = O.sigmoid_fwd(want)
    elif act_end == ACT_LEAKY:
        want = O.leaky_relu_fwd(want, alpha_end)
    return want


def test_line_network_one_kernel_vs_oracle(nn):
    """uocr_hourglass4_fwd: the whole Line network (1 -> 4 -> 4 -> 4 -> 4 -> 2 channels) as ONE tensor-core kernel
    (csrc/hourglass4_tc.cu) vs the float64 oracle chain of five conv layers, through the C ABI with raw pointers: the
    Line tile (2, 128, 256), sizes that end inside a 16 x 128 block, sizes smaller than one block, a page-wide strip, and
    every end activation.  Signed weights (un-saturated sigmoids); tolerance 1e-3 of the output range for the sigmoid
    output, 2e-3 for the un-squashed outputs (five layers of gain).  The packed-weights entry gives the same bits."""
    import ctypes
    from univer_ocr_b200._lib import ACT_LEAKY, ACT_NONE, ACT_SIGMOID, lib
    rng = np.random.default_rng(77)
    ptrs = ctypes.c_void_p * 5
    for (n, h, w), act_end in (((2, 128, 256), ACT_SIGMOID), ((1, 16, 128), ACT_NONE), ((3, 4, 4), ACT_SIGMOID),
                               ((2, 20, 36), ACT_LEAKY), ((1, 52, 300), ACT_SIGMOID), ((1, 132, 12), ACT_NONE),
                               ((2, 8, 2064), ACT_SIGMOID), ((1, 496, 736), ACT_SIGMOID)):
        X = f32(rng.uniform(size=(n, h, w, 1)))
        chans = [(1, 4), (4, 4), (4, 4), (4, 4), (4, 2)]
        ws = [f32(rng.standard_normal((5, 5, ci, co)) * (0.6 / np.sqrt(ci * 6.0))) for ci, co in chans]
        bs = [f32(rng.standard_normal(co) * 0.2) for _, co in chans]
        want = _line_oracle(X, ws, bs, act_end, alpha_end=0.2)
        dX, dw, db = nn.CP.copy(X), [nn.CP.copy(a) for a in ws], [nn.CP.copy(a) for a in bs]
        y = nn.DeviceArray.full((n, h, w, 2), -3.0)
        lib.uocr_hourglass4_fwd(dX.ptr, ptrs(*[a.ptr for a in dw]), ptrs(*[a.ptr for a in db]), y.ptr, n, h, w,
                                0.01, act_end, 0.2, nn.CP.stream())
        got = np.asarray(y.get(), dtype=np.float64)
        assert np.isfinite(got).all()
        if act_end == ACT_SIGMOID:
            assert 0.05 < want.mean() < 0.95 and want.std() > 0.02, 'saturated test case'
        close_tf32(got, want, f'line one-kernel vs oracle {(n, h, w)}', tol=1e-3 if act_end == ACT_SIGMOID else 2e-3)
        count = ctypes.c_int64()
        lib.uocr_hourglass4_packed_floats(ctypes.byref(count))
        packed = nn.DeviceArray((count.value,))
        lib.uocr_hourglass4_pack(ptrs(*[a.ptr for a in dw]), packed.ptr, nn.CP.stream())
        y2 = nn.DeviceArray.full((n, h, w, 2), -3.0)
        lib.uocr_hourglass4_fwd_packed(dX.ptr, packed.ptr, ptrs(*[a.ptr for a in db]), y2.ptr, n, h, w, 0.01, act_end, 0.2,
                                       nn.CP.stream())
        assert np.array_equal(y2.get(), y.get())
    # error convention: geometry the kernel does not implement
    from univer_ocr_b200._lib import UocrError
    with pytest.raises(UocrError) as err:
        lib.uocr_hourglass4_fwd(dX.ptr, ptrs(*[a.ptr for a in dw]), ptrs(*[a.ptr for a in db]), y.ptr, 1, 6, 8,
                                0.01, ACT_SIGMOID, 0.0, nn.CP.stream())
    assert err.value.code == -3 and 'multiples of 4' in str(err.value)


def test_line_model_uses_the_one_kernel_path(nn):
    """my_model.make_line in TF32 mode: Model.predict goes through HourglassFusion -> uocr_hourglass4_fwd_packed (one
    launch + one pack launch on the first call / after a weight change) and agrees with the layer-by-layer FP32 path;
    in FP32 mode the fusion steps aside."""
    from univer_ocr_b200 import my_model
    from univer_ocr_b200._lib import launch_count
    shape = (2, 128, 256, 1)
    model = my_model.make_line(shape)
    for key, p in model.params().items():                                 # centred: the default init saturates the sigmoid
        v = np.asarray(p.value.get(), dtype=np.float64)
        p.value = (v - v.mean()) * 3.5 if v.size > 2 else v * 0.25
    x = f32(np.random.default_rng(3).uniform(size=shape))
    nn.CP.set_math_mode('tf32')
    try:
        assert model.infer_fusion is not None
        n0 = launch_count()
        y1 = model.predict(x)[0].get()
        first = launch_count() - n0
        n0 = launch_count()
        y2 = model.predict(x)[0].get()
        second = launch_count() - n0
        assert np.array_equal(y1, y2)
        assert second == 1 and first == 2, (first, second)
        # a weight change re-packs
        for key, p in model.params().items():
            if key.endswith('end/conv_1/w'):
                p.value = np.asarray(p.value.get()) * 0.5
        y3 = model.predict(x)[0].get()
        assert not np.array_equal(y1, y3)
        nn.CP.set_math_mode('fp32')
        n0 = launch_count()
        ref = model.predict(x)[0].get()
        assert launch_count() - n0 >= 5                                # layer by layer
    finally:
        nn.CP.set_math_mode('tf32')
    assert 0.05 < ref.mean() < 0.95
    close_tf32(np.asarray(y3, dtype=np.float64), np.asarray(ref, dtype=np.float64), 'line model fused vs fp32', tol=1e-3)


@pytest.mark.parametrize('batch,n_in,n_hidden,n_out,mode', [
    (16384, 1024, 128, 162, 'tf32'),     # Char dense_2 + leaky_relu_2 + dense_3 at batch 64: the one-kernel path
    (1000, 1024, 128, 162, 'tf32'),      # ragged last tile
    (4096, 64, 128, 16, 'tf32'), (640, 256, 128, 256, 'tf32'), (777, 128, 128, 200, 'tf32'),
    (300, 96, 64, 30, 'tf32'),           # hidden width the kernel is not built for: two GEMMs inside the library
    (200, 50, 128, 162, 'tf32'),         # n_in % 32 != 0: likewise
    (300, 1024, 128, 162, 'fp32'),       # FP32 check mode: likewise, FFMA
])
def test_fc_chain_vs_oracle(nn, batch, n_in, n_hidden, n_out, mode):
    """uocr_fc_chain2_fwd: FullyConnected + LeakyRelu + FullyConnected (make_dense_block, my_model/model.py:251-262) in
    one call vs the float64 oracle (layers.py:335-347 twice); the one-kernel path keeps the hidden tile in shared memory
    in the tensor-core operand layout.  TF32: 1e-3 of the output range per GEMM -> 2e-3; FP32: 1e-4."""
    from univer_ocr_b200._lib import ACT_LEAKY, MATH_FP32, MATH_TF32, lib
    rng = np.random.default_rng(batch + n_in + n_out)
    X = f32(rng.standard_normal((batch, n_in)))
    W1 = f32(rng.standard_normal((n_in + 1, n_hidden)) / np.sqrt(n_in))
    W2 = f32(rng.standard_normal((n_hidden + 1, n_out)) / np.sqrt(n_hidden))
    want = O.fc_fwd(O.leaky_relu_fwd(O.fc_fwd(X, W1), 0.01), W2)
    dX, dW1, dW2 = nn.CP.copy(X), nn.CP.copy(W1), nn.CP.copy(W2)
    y = nn.DeviceArray.full((batch, n_out), -7.0)
    for kmajor in (False, True):
        w1t = w2t = None
        if kmajor:
            w1t, w2t = nn.DeviceArray((n_hidden, n_in)), nn.DeviceArray((n_out, n_hidden))
            lib.uocr_weights_to_kmajor(dW1.ptr, w1t.ptr, n_in, n_hidden, nn.CP.stream())
            lib.uocr_weights_to_kmajor(dW2.ptr, w2t.ptr, n_hidden, n_out, nn.CP.stream())
        lib.uocr_fc_chain2_fwd(dX.ptr, dW1.ptr, w1t.ptr if kmajor else None, dW2.ptr, w2t.ptr if kmajor else None, y.ptr,
                               batch, n_in, n_hidden, n_out, ACT_LEAKY, 0.01, MATH_TF32 if mode == 'tf32' else MATH_FP32,
                               nn.CP.stream())
        got = np.asarray(y.get(), dtype=np.float64)
        if mode == 'tf32':
            close_tf32(got, want, f'fc chain {(batch, n_in, n_hidden, n_out)} kmajor={kmajor}', tol=2e-3)
        else:
            assert np.abs(got - want).max() <= 1e-4 * np.abs(want).max()


def test_char_head_runs_as_two_launches(nn):
    """Inference plan of make_char in TF32 mode: window batching + Flatten + dense_1 + LeakyRelu is one GEMM, dense_2 +
    LeakyRelu + dense_3 one kernel -- 5 launches for the whole network -- and agrees with the layer-by-layer plan."""
    from oracle import np_models
    from univer_ocr_b200 import my_model
    from univer_ocr_b200._lib import launch_count
    shape = (64, 32, 256, 1)
    w0 = np_models.golden_weights('char', 5)
    X = nn.CP.copy(f32(np.random.default_rng(1).uniform(size=shape)))
    nn.CP.set_math_mode('tf32')
    model = my_model.make_char(shape)
    model.set_weights({k: {n: v.tolist() for n, v in p.items()} for k, p in w0.items()})
    assert [s[0] for s in model._plan_infer] == ['conv', 'conv', 'conv', 'winfc', 'fcchain']
    fused = model.predict(X)[0].get()
    n0 = launch_count()
    model.predict(X)
    assert launch_count() - n0 == 5
    model.fusion = False
    model.initialize(model.input_shapes)
    plain = model.predict(X)[0].get()
    assert np.abs(fused - plain).max() <= 2e-3 * np.abs(plain).max()
