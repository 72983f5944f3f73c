"""Ragged batches: images of different sizes on one zero-filled canvas (include/uocr.h, Model.predict_ragged,
TextPipeline.batch).  The CPU tests cover the host-side analysis; the GPU tests compare every ragged path with the
same work done one image at a time."""
import ctypes

import numpy as np
import pytest

from tests import stage_cases as C


def _tol_ok(got, want, tf32):
    """DESIGN.md §4: FP32 rtol 1e-4 + 2e-6 * max|want|, TF32 1e-3 of the output range."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    if tf32:
        span = max(float(want.max() - want.min()), 1e-30)
        return np.abs(got - want).max() <= 1e-3 * span
    return np.all(np.abs(got - want) <= 1e-4 * np.abs(want) + 2e-6 * np.abs(want).max())


# ---------------------------------------------------------------------------------------------- host side

def test_ragged_extents_match_per_image_shape_analysis():
    """Per-image output extents = get_output_shapes of (1, h_i, w_i, C) for all four networks; Char's rows are
    [i * W, i * W + w_i) of the (N * W, classes) output."""
    from univer_ocr_b200 import my_model
    rng = np.random.default_rng(0)
    for name, (h, w) in (('monochrome', (40, 52)), ('paragraph', (48, 64)), ('line', (64, 96)), ('char', (32, 120))):
        n = 7
        model = my_model.MAKERS[name]((n, h, w, 1))
        hs = np.full(n, h) if name == 'char' else rng.integers(1, h + 1, n)
        ws = rng.integers(8, w + 1, n)
        hs[0], ws[0] = h, w
        ext = np.stack([hs, ws], axis=1)
        _, modes = model.ragged_analysis((n, h, w, 1), ext)
        out = model.relations[0][0]
        kind, table, _ = modes[out]
        for i, (eh, ew) in enumerate(ext):
            want = model.get_output_shapes([(1, int(eh), int(ew), 1)])[0]
            if name == 'char':
                assert kind == 'rows' and tuple(table[i]) == (i * w, i * w + ew) and want[0] == ew
            else:
                assert kind == 'hw' and tuple(table[i]) == want[1:3]


def test_predict_ragged_rejects_bad_input_before_launching():
    """Out-of-range extents, a wrong table shape, MaxPool2D and a conv with padding_value != 0 raise ValueError in the
    host analysis, i.e. before anything is uploaded or launched (these run without a device)."""
    from univer_ocr_b200 import my_model
    from univer_ocr_b200.nn.layers import Convolutional2D, MaxPool2D
    from univer_ocr_b200.nn.models import Sequential
    model = my_model.make_monochrome((2, 16, 16, 1))
    for bad in ([[0, 4], [16, 16]], [[4, 17], [16, 16]], [[17, 4], [1, 1]], [[4, 4]], [[1.5, 2], [3, 4]]):
        with pytest.raises(ValueError):
            model.predict_ragged(np.zeros((2, 16, 16, 1), np.float32), np.array(bad))
    for layers, what in (([MaxPool2D(2)], 'MaxPool2D'), ([Convolutional2D(3, out_channels=2, padding=1, padding_value=1.0)],
                                                         'padding_value')):
        seq = Sequential(layers)
        seq.initialize((2, 16, 16, 1))
        with pytest.raises(ValueError, match=what):
            seq.predict_ragged(np.zeros((2, 16, 16, 1), np.float32), np.array([[8, 8], [16, 16]]))


# ---------------------------------------------------------------------------------------------- device

@pytest.fixture(scope='module')
def nn():
    import univer_ocr_b200.nn as nn_
    nn_.CP.use_gpu()
    keep = nn_.CP.math_mode
    yield nn_
    nn_.CP.math_mode = keep


def _dev_ext(nn, ext):
    return nn.DeviceArray.from_host(np.asarray(ext, np.int32), np.int32)


@pytest.mark.gpu
def test_zero_pack_unpack_match_numpy(nn):
    """uocr_zero_outside_hw_f32, uocr_pack_hw_f32, uocr_unpack_hw_f32: bit-exact against NumPy for C in {1, 2, 4, 64},
    extents incl. 1 x 1, the whole canvas and widths that are not multiples of 4; extents beyond the canvas are clamped
    and nothing outside the canvas is written."""
    from univer_ocr_b200._lib import lib
    rng = np.random.default_rng(1)
    for c in (1, 2, 4, 64):
        n, h, w = 6, 13, 23
        ext = np.array([[1, 1], [h, w], [5, 7], [13, 3], [2, 22], [9, 17]])
        x = rng.standard_normal((n, h, w, c)).astype(np.float32)
        want = x.copy()
        for i, (eh, ew) in enumerate(ext):
            want[i, eh:] = 0
            want[i, :, ew:] = 0
        guard = 1000
        buf = nn.DeviceArray.from_host(np.full(x.size + 2 * guard, 7.0, np.float32))
        dx = buf.flat_view(guard, x.size, x.shape)
        dx.set(x)
        de = _dev_ext(nn, ext)
        lib.uocr_zero_outside_hw_f32(dx.ptr, de.ptr, n, h, w, c, nn.CP.stream())
        assert np.array_equal(dx.get(), want), c
        images = [rng.standard_normal((1, eh, ew, c)).astype(np.float32) for eh, ew in ext]
        dimg = [nn.CP.copy(a) for a in images]
        canvas = buf.flat_view(guard, x.size, x.shape)
        lib.uocr_pack_hw_f32((ctypes.c_void_p * n)(*[a.ptr for a in dimg]), de.ptr, canvas.ptr, n, h, w, c,
                             nn.CP.stream())
        packed = np.zeros_like(x)
        for i, a in enumerate(images):
            packed[i, :a.shape[1], :a.shape[2]] = a
        assert np.array_equal(canvas.get(), packed), c
        outs = [nn.DeviceArray.zeros(a.shape) for a in images]
        lib.uocr_unpack_hw_f32(canvas.ptr, de.ptr, (ctypes.c_void_p * n)(*[o.ptr for o in outs]), n, h, w, c,
                               nn.CP.stream())
        for o, a in zip(outs, images):
            assert np.array_equal(o.get(), a), c
        # out-of-range extents: clamped to the canvas, the guard bands stay untouched
        wild = _dev_ext(nn, [[h + 50, w + 9], [-3, 4], [2, 10 ** 6], [0, 0], [h, w], [1, -1]])
        lib.uocr_zero_outside_hw_f32(canvas.ptr, wild.ptr, n, h, w, c, nn.CP.stream())
        full = buf.get()
        assert (full[:guard] == 7.0).all() and (full[guard + x.size:] == 7.0).all()


@pytest.mark.gpu
def test_ragged_line_kernel_bit_identical_per_image(nn):
    """Model.predict_ragged of the Line network (TF32: uocr_hourglass4_fwd_packed_ragged) == Model.predict on every
    image alone (uocr_hourglass4_fwd_packed), bit for bit, and 0 outside each extent; ~20 images with extents that are
    multiples of 4 and of 16, one equal to the canvas, a canvas larger than the other extents."""
    from univer_ocr_b200 import my_model
    from univer_ocr_b200._lib import launch_count
    nn.CP.set_math_mode('tf32')
    rng = np.random.default_rng(2)
    n, h, w = 20, 96, 272
    ext = np.stack([rng.integers(1, h // 4 + 1, n) * 4, rng.integers(1, w // 4 + 1, n) * 4], axis=1)
    ext[1] = (h, w)
    ext[2] = (16, 32)
    ext[3] = (4, 4)
    model = my_model.make_line((n, h, w, 1))
    canvas = np.zeros((n, h, w, 1), np.float32)
    images = []
    for i, (eh, ew) in enumerate(ext):
        images.append(rng.uniform(0, 1, (1, eh, ew, 1)).astype(np.float32))
        canvas[i, :eh, :ew] = images[i]
    before = launch_count()
    outs, out_ext = model.predict_ragged(nn.CP.copy(canvas), ext)
    got = outs[0].get()
    assert launch_count() - before <= 2                 # the ragged kernel (+ the weight packing on the first call)
    assert np.array_equal(out_ext[0], ext)
    for i, (eh, ew) in enumerate(ext):
        want = model.predict(nn.CP.copy(images[i]))[0].get()
        assert np.array_equal(got[i:i + 1, :eh, :ew], want), i
        assert not got[i, eh:].any() and not got[i, :, ew:].any(), i


@pytest.mark.gpu
@pytest.mark.parametrize('mode', ['fp32', 'tf32'])
@pytest.mark.parametrize('name', ['monochrome', 'paragraph', 'line', 'char'])
def test_predict_ragged_matches_predict_per_image(nn, name, mode):
    """Model.predict_ragged == Model.predict on each image alone, within the tolerances of DESIGN.md §4.  Char with
    every line as wide as the canvas runs the same kernels on both sides: bit-identical."""
    from univer_ocr_b200 import my_model
    nn.CP.set_math_mode(mode)
    rng = np.random.default_rng(3)
    n, h, w = 5, (32 if name == 'char' else 48), (96 if name == 'char' else 80)
    if name == 'char':
        ext = np.stack([np.full(n, h), rng.integers(8, w + 1, n)], axis=1)
    else:
        ext = np.stack([rng.integers(4, h + 1, n), rng.integers(4, w + 1, n)], axis=1)
    ext[0] = (h, w)
    if name == 'line':
        ext[1] = (20, 36)                                   # multiples of 4 (TF32: the ragged kernel) ...
        ext[2] = (18, 30)                                   # ... and not (the layer plan with masks)
    model = my_model.MAKERS[name]((n, h, w, 1))
    canvas = np.zeros((n, h, w, 1), np.float32)
    images = []
    for i, (eh, ew) in enumerate(ext):
        images.append(rng.uniform(0, 1, (1, eh, ew, 1)).astype(np.float32))
        canvas[i, :eh, :ew] = images[i]
    outs, out_ext = model.predict_ragged(nn.CP.copy(canvas), ext)
    got = outs[0].get()
    for i in range(n):
        want = model.predict(nn.CP.copy(images[i]))[0].get()
        if name == 'char':
            a, b = out_ext[0][i]
            part = got[a:b]
        else:
            oh, ow = out_ext[0][i]
            part = got[i:i + 1, :oh, :ow]
            assert not got[i, oh:].any() and not got[i, :, ow:].any()
        assert part.shape == want.shape, (name, i)
        assert _tol_ok(part, want, mode == 'tf32'), (name, mode, i)
    if name == 'char':
        full = np.stack([np.full(n, h), np.full(n, w)], axis=1)
        outs, _ = model.predict_ragged(nn.CP.copy(canvas), full)
        assert np.array_equal(outs[0].get(), model.predict(nn.CP.copy(canvas))[0].get())


def _standins(nn, pages_pred):
    from univer_ocr_b200 import my_model

    def lines_for(shape):
        _, h, w, _ = shape
        out = np.zeros((1, h, w, 2), np.float32)
        for centre in (h // 3, (2 * h) // 3):
            out[0, centre - 6:centre - 4, 6:w - 6, 0] = 1.0
            out[0, centre + 4:centre + 6, 6:w - 6, 1] = 1.0
        return out

    def chars_for(line):
        cols = np.asarray(line)[0, :, :, 0].mean(axis=0)
        out = np.zeros((cols.size, my_model.N_CHARS), np.float32)
        out[np.arange(cols.size), (cols * 40).astype(int) % my_model.N_CHARS] = 1.0
        return out

    def paragraph(x):
        return nn.CP.copy(pages_pred[tuple(x.shape)])

    return {'monochrome': lambda x: x, 'paragraph': paragraph,
            'line': lambda x: nn.CP.copy(lines_for(x.shape)), 'char': lambda x: nn.CP.copy(chars_for(x.get()))}


def _same_result(got, want):
    assert got['text'] == want['text'] and got['angles'] == want['angles']
    for key in ('monochrome_pred', 'paragraph_pred'):
        assert np.array_equal(got[key].get(), want[key].get())
    for g, w in zip(got['cropped_monochrome'], want['cropped_monochrome']):
        assert np.array_equal(g.get(), w.get())
    assert len(got['cropped_monochrome']) == len(want['cropped_monochrome'])
    assert [len(p) for p in got['cropped_2_monochrome']] == [len(p) for p in want['cropped_2_monochrome']]
    for gp, wp in zip(got['cropped_2_monochrome'], want['cropped_2_monochrome']):
        for g, w in zip(gp, wp):
            assert np.array_equal(g.get(), w.get())


@pytest.mark.gpu
def test_text_pipeline_batch_with_standins_equals_per_page(nn):
    """TextPipeline.batch == [pipe(page) for page in pages] with deterministic stand-ins: three pages of different sizes
    and paragraph counts, one with nothing to cut -- text, angles and crops bit for bit."""
    from oracle import np_oracle as O
    from univer_ocr_b200 import my_model, predict
    pred_a, images_a = C.paragraph_page(3, h=150, w=230)
    pred_b, images_b = C.paragraph_page(1, h=160, w=240, tilt=(80.0, 3.0))
    pages = [images_a[0], images_b[0], np.zeros((1, 40, 60, 1), np.float32)]
    preds = {}
    for pred, page in ((pred_a, pages[0]), (pred_b, pages[1])):
        padded = O.make_divisible_by(pred, 16, 16).astype(np.float32)
        preds[tuple(O.make_divisible_by(page, 16, 16).shape)] = padded
    preds[(1, 48, 64, 1)] = np.full((1, 48, 64, 1), 0.25, np.float32)
    chars = [chr(33 + i) for i in range(my_model.N_CHARS)]
    pipe = predict.TextPipeline(predictors=_standins(nn, preds), chars=chars, are_similar=lambda a, b: a == b)
    want = [pipe(p) for p in pages]
    got = pipe.batch(pages)
    assert len(got) == 3 and want[2]['text'] == [] and sum(len(w['text']) for w in want) >= 3
    for g, w in zip(got, want):
        _same_result(g, w)


@pytest.mark.gpu
def test_text_pipeline_batch_runs_line_and_char_once(nn):
    """TextPipeline.batch with the real Char network: one Char call per batch (Model.predict_ragged), one network
    instance whose weights are uploaded once, per-line char_pred within tolerance of the per-page path, hits identical
    wherever the per-page top-2 margin exceeds twice the tolerance.  The batch's Line step with the real Line network
    (one ragged call over every paragraph of the batch, unpacked per paragraph) equals Line on each paragraph alone, bit
    for bit.  (An untrained Line network marks no lines, so the batch itself reads lines marked by a stand-in.)"""
    from oracle import np_oracle as O
    from univer_ocr_b200 import predict
    from univer_ocr_b200.nn import models
    nn.CP.set_math_mode('tf32')
    pred_a, images_a = C.paragraph_page(3, h=150, w=230)
    pred_b, images_b = C.paragraph_page(0, h=160, w=240)
    preds = {tuple(O.make_divisible_by(p, 16, 16).shape): O.make_divisible_by(q, 16, 16).astype(np.float32)
             for p, q in ((images_a[0], pred_a), (images_b[0], pred_b))}
    stand = _standins(nn, preds)
    pipe = predict.TextPipeline(predictors={k: stand[k] for k in ('monochrome', 'paragraph', 'line')})
    calls = []
    orig = models.Model.predict_ragged

    def counting(self, canvas, extents):
        calls.append(self)
        return orig(self, canvas, extents)

    models.Model.predict_ragged = counting
    try:
        got = pipe.batch([images_a[0], images_b[0]])
        assert len(calls) == 1 and set(pipe._models) == {'char'}
        char_model = pipe._models['char']
        weights = [p.value.ptr for p in char_model.params().values()]
        want = [pipe(p) for p in (images_a[0], images_b[0])]
        assert pipe._models['char'] is char_model
        assert [p.value.ptr for p in char_model.params().values()] == weights        # no re-upload for new shapes
        n_lines = 0
        for g, w in zip(got, want):
            assert [len(p) for p in g['char_pred']] == [len(p) for p in w['char_pred']]
            for gp, wp in zip(g['char_pred'], w['char_pred']):
                for gl, wl in zip(gp, wp):
                    a, b = gl.get(), wl.get()
                    assert a.shape == b.shape and _tol_ok(a, b, True)
                    tol = 1e-3 * float(b.max() - b.min())
                    top2 = np.sort(b, axis=1)[:, -2:]
                    wide = (top2[:, 1] - top2[:, 0]) > 2 * tol
                    hits_a = a[wide] == a[wide].max(axis=1, keepdims=True)
                    hits_b = b[wide] == b[wide].max(axis=1, keepdims=True)
                    assert np.array_equal(hits_a, hits_b)
                    n_lines += 1
        assert n_lines >= 4
        # the batch's Line step with the real network
        del pipe.predictors['line']
        crops = [t for g in got for t in g['cropped_monochrome']]
        calls.clear()
        line_pred = pipe._unpack(*pipe._ragged('line', crops))
        assert len(calls) == 1 and len(crops) >= 3
        line_model = pipe._models['line']
        for crop, lp in zip(crops, line_pred):
            assert np.array_equal(lp.get(), pipe.predict('line', crop).get())
        assert pipe._models['line'] is line_model
    finally:
        models.Model.predict_ragged = orig
