"""Ragged training batches: one training step over images of different sizes on one zero-filled canvas
(include/uocr.h uocr_seg_loss_ragged / uocr_seg_grad_ragged / uocr_softmax_ce_rows, Model.train_ragged,
DataParallel.train_ragged, Trainer).  The CPU tests cover the host-side checks and the Trainer's packing; the GPU tests
compare every ragged path with the same work done one image at a time."""
import os
import sys

import numpy as np
import pytest

from tests import trainer_cases

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------------------------------------- host side

def test_ragged_train_analysis_rejects_bad_input_before_launching():
    """An unsupported loss, a target of the wrong shape or row count, padding_value != 0 and an extent outside the
    canvas raise ValueError in the host analysis, before anything is uploaded or launched (these run without a
    device)."""
    from univer_ocr_b200 import my_model
    from univer_ocr_b200.nn.layers import Convolutional2D, Sigmoid
    from univer_ocr_b200.nn.losses import SegmentationDice2D, SigmoidCrossEntropy
    from univer_ocr_b200.nn.models import Sequential
    canvas = np.zeros((2, 16, 16, 1), np.float32)
    ext = np.array([[8, 12], [16, 16]])

    def rejects(model, c, e, y, match):
        for call in (model.compute_loss_and_gradients_ragged, model.train_ragged, model.test_ragged):
            with pytest.raises(ValueError, match=match):
                call(c, e, y)

    seq = Sequential([Convolutional2D(3, out_channels=1, padding=1), Sigmoid()], loss=SigmoidCrossEntropy())
    seq.initialize((2, 16, 16, 1))
    rejects(seq, canvas, ext, np.zeros((2, 16, 16, 1), np.float32), 'SigmoidCrossEntropy')
    seq = Sequential([Convolutional2D(3, out_channels=1, padding=1, padding_value=1.0), Sigmoid()],
                     loss=SegmentationDice2D())
    seq.initialize((2, 16, 16, 1))
    rejects(seq, canvas, ext, np.zeros((2, 16, 16, 1), np.float32), 'padding_value')

    mono = my_model.make_monochrome((2, 16, 16, 1))
    rejects(mono, canvas, ext, np.zeros((2, 16, 15, 1), np.float32), 'target of shape')
    rejects(mono, canvas, ext, [np.zeros((2, 16, 16, 1), np.float32)] * 2, 'targets for')
    rejects(mono, canvas, np.array([[8, 17], [16, 16]]), np.zeros((2, 16, 16, 1), np.float32), 'outside')
    rejects(mono, canvas, np.array([[0, 4], [16, 16]]), np.zeros((2, 16, 16, 1), np.float32), 'outside')

    char = my_model.make_char((2, 32, 20, 1))
    y_rows = np.zeros((2 * 20, my_model.N_CHARS), np.float32)
    for bad in (y_rows[:-1], np.zeros((2 * 20, my_model.N_CHARS - 1), np.float32)):
        rejects(char, np.zeros((2, 32, 20, 1), np.float32), np.array([[32, 9], [32, 20]]), bad, 'target of shape')


class _RaggedModel(trainer_cases.ScriptedModel):
    """A scripted model that records which step each batch reached and with what."""

    def __init__(self, name, w0, optimizer, mean=False):
        super().__init__(name, w0, optimizer)
        self.mean_over_batch = mean
        self.calls = []

    def train(self, X, y):
        self.calls.append(('train', np.asarray(X), np.asarray(y), None, None))
        return super().train(X, y)

    def test(self, X, y):
        self.calls.append(('test', np.asarray(X), np.asarray(y), None, None))
        return super().test(X, y)

    def train_ragged(self, canvas, extents, y, rows_total=None):
        self.calls.append(('train_ragged', np.asarray(canvas), np.asarray(y), np.asarray(extents), rows_total))
        return super().train(canvas, y)

    def test_ragged(self, canvas, extents, y):
        self.calls.append(('test_ragged', np.asarray(canvas), np.asarray(y), np.asarray(extents), None))
        return super().test(canvas, y)


class _SizedDataset:
    """Sample i: X (1, h_i, w_i, 1) in [0.1, 1) and y either an image map (1, h_i, w_i, 1) or w_i rows of 3 classes."""

    def __init__(self, sizes, rows, seed):
        rng = np.random.default_rng(seed)
        self.samples = []
        for h, w in sizes:
            X = rng.uniform(0.1, 1.0, (1, h, w, 1))
            y = rng.uniform(0.1, 1.0, (w, 3) if rows else (1, h, w, 1))
            self.samples.append({'m': (X, y)})

    def __len__(self):
        return len(self.samples)

    def get(self, i):
        return self.samples[i]


def _trainer(model, train_ds, val_ds, batch_size, **kwargs):
    from univer_ocr_b200.trainer import Trainer
    return Trainer({'m': model}, train_ds, val_ds, optimizer=model.optimizer, batch_size=batch_size,
                   shuffle=lambda order: None, log=lambda *a, **k: None, **kwargs)


@pytest.mark.parametrize('rows', [False, True])
def test_trainer_packs_mixed_size_samples_on_a_canvas(rows):
    """Mixed-size samples reach train_ragged / test_ragged with X on a zero-filled canvas, one (h, w) row per image, and
    y on its canvas (image maps) or at rows [i * W, i * W + w_i) (window rows); same-size batches still reach train /
    test, stacked."""
    sizes = [(5, 9), (7, 4), (2, 11), (7, 6)]
    train_ds = _SizedDataset(sizes + [(3, 3), (3, 3)], rows, 1)
    val_ds = _SizedDataset([(4, 4), (4, 4)], rows, 2)
    model = _RaggedModel('m', 0.5, trainer_cases.ScriptedOptimizer(0.0), mean=rows)
    _trainer(model, train_ds, val_ds, batch_size=4, prefetch=0).train(1)
    kinds = [c[0] for c in model.calls]
    assert kinds == ['test', 'train_ragged', 'train', 'test']
    _, canvas, y, ext, rows_total = model.calls[1]
    assert rows_total is None
    H, W = max(h for h, _ in sizes), max(w for _, w in sizes)
    assert canvas.shape == (4, H, W, 1) and canvas.dtype == np.float32
    assert np.array_equal(ext, np.array(sizes))
    for i, (h, w) in enumerate(sizes):
        X_i, y_i = train_ds.get(i)['m']
        assert np.array_equal(canvas[i, :h, :w], X_i[0].astype(np.float32))
        assert not canvas[i, h:].any() and not canvas[i, :, w:].any()
        if rows:
            assert y.shape == (4 * W, 3)
            assert np.array_equal(y[i * W:i * W + w], y_i.astype(np.float32))
            assert not y[i * W + w:(i + 1) * W].any()
        else:
            assert y.shape == (4, H, W, 1)
            assert np.array_equal(y[i, :h, :w], y_i[0].astype(np.float32))
            assert not y[i, h:].any() and not y[i, :, w:].any()
    _, X, _, _, _ = model.calls[2]
    assert X.shape == (2, 3, 3, 1)


def _two_rank_ragged_worker(rank, world, port, out):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ['MASTER_ADDR'], os.environ['MASTER_PORT'] = '127.0.0.1', str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from tests.gloo_comm import GlooComm
    # rank 0 trains samples 0 and 2 (widths 9 and 4: ragged), rank 1 samples 1 and 3 (both 6 wide: stackable)
    train_ds = _SizedDataset([(5, 9), (5, 6), (5, 4), (5, 6)], True, 3)
    val_ds = _SizedDataset([(5, 5), (5, 7)], True, 4)
    model = _RaggedModel('m', 0.5, trainer_cases.ScriptedOptimizer(0.0), mean=True)
    comm = GlooComm()
    _trainer(model, train_ds, val_ds, batch_size=4, prefetch=0, comm=comm).train(1)
    out.put((rank, [(c[0], None if c[3] is None else c[3].tolist(), c[4]) for c in model.calls]))
    dist.destroy_process_group()


def test_two_ranks_sum_valid_rows_for_mean_losses():
    """gloo world size 2, a mean-over-batch model: rank 0's batch is ragged and rank 1's is not; both ranks take the
    ragged step (rank 1 with its stacked batch as a canvas without padding) and get rows_total = the valid rows of both
    ranks (9 + 4 + 6 + 6); validation steps (one sample per rank) stay local."""
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    out = ctx.Queue()
    port = 29600 + os.getpid() % 90
    procs = [ctx.Process(target=_two_rank_ragged_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    got = dict(out.get(timeout=10) for _ in range(2))
    assert [c[0] for c in got[0]] == [c[0] for c in got[1]] == ['test', 'train_ragged', 'test']
    assert got[0][1][1:] == ([[5, 9], [5, 4]], 25) and got[1][1][1:] == ([[5, 6], [5, 6]], 25)


# ---------------------------------------------------------------------------------------------- device

@pytest.fixture(scope='module')
def nn():
    import univer_ocr_b200.nn as nn_
    nn_.CP.use_gpu()
    keep = nn_.CP.math_mode
    yield nn_
    nn_.CP.math_mode = keep


def _dev_i32(nn, table):
    return nn.DeviceArray.from_host(np.asarray(table, np.int32), np.int32)


def _view(nn, host, offset):
    """A device copy of `host` starting `offset` floats into its buffer (offset 1: not 16-byte aligned)."""
    buf = nn.DeviceArray.zeros((host.size + 4,))
    v = buf.flat_view(offset, host.size, host.shape)
    v.set(np.ascontiguousarray(host, np.float32))
    return v


SEG_EXTENTS = np.array([[1, 1], [13, 23], [5, 7], [13, 3], [2, 22], [9, 17]])


@pytest.mark.gpu
@pytest.mark.parametrize('offset', [0, 1])
@pytest.mark.parametrize('c', [1, 2])
@pytest.mark.parametrize('kind', [0, 1])
def test_seg_loss_ragged_matches_float64(nn, kind, c, offset):
    """uocr_seg_loss_ragged and uocr_seg_grad_ragged (with and without x_pre) against NumPy float64: extents from 1 x 1
    to the whole 13 x 23 canvas, widths that are not multiples of 4, 16-byte aligned and unaligned views.  NaN outside
    every extent in pred, gt and x_pre shows nothing there is read; the gradient is exactly 0 there."""
    import ctypes
    from univer_ocr_b200._lib import lib
    rng = np.random.default_rng(10 + kind + 2 * c)
    n, (h, w) = len(SEG_EXTENTS), SEG_EXTENTS.max(axis=0)
    pred = rng.uniform(0.01, 0.99, (n, h, w, c)).astype(np.float32)
    gt = (rng.uniform(size=(n, h, w, c)) < 0.4).astype(np.float32)
    xpre = rng.uniform(-4, 4, (n, h, w, c)).astype(np.float32)
    inside = np.zeros((n, h, w, c), bool)
    for i, (eh, ew) in enumerate(SEG_EXTENTS):
        inside[i, :eh, :ew] = True
    for a in (pred, gt, xpre):
        a[~inside] = np.nan
    eps = 1e-8
    p, g = np.where(inside, pred, 0).astype(np.float64), np.where(inside, gt, 0).astype(np.float64)
    num = (p * g).sum(axis=(1, 2)) + eps
    sp, sg = p.sum(axis=(1, 2)), g.sum(axis=(1, 2))
    if kind == 0:
        den = sp + sg + 2 * eps
        loss, a, b = (1 - 2 * num / den).sum(), -2 / den, 2 * num / den ** 2
    else:
        den = sp + sg - num + 2 * eps
        loss, a, b = (1 - num / den).sum(), -(den + num) / den ** 2, num / den ** 2
    want = np.where(inside, a[:, None, None, :] * g + b[:, None, None, :], 0)
    x64 = np.where(inside, xpre, 0).astype(np.float64)
    want_sig = want * np.exp(-x64) / (1 + np.exp(-x64)) ** 2

    need = ctypes.c_size_t(0)
    lib.uocr_seg_loss_workspace(n, c, ctypes.byref(need))
    ws = nn.DeviceArray(((need.value + 7) // 8,), 'float64')
    d_pred, d_gt, d_x = _view(nn, pred, offset), _view(nn, gt, offset), _view(nn, xpre, offset)
    d_ext = _dev_i32(nn, SEG_EXTENTS)
    d_loss = nn.DeviceArray.zeros((1,))
    grad = _view(nn, np.full(pred.shape, 7.0, np.float32), offset)
    lib.uocr_seg_loss_ragged(kind, d_pred.ptr, d_gt.ptr, grad.ptr, d_loss.ptr, d_ext.ptr, n, h, w, c, ws.ptr,
                             nn.CP.stream())
    got = grad.get()
    assert abs(float(d_loss.get()[0]) - loss) <= 1e-5 * abs(loss)
    assert not got[~inside].any()
    assert np.abs(got - want).max() <= 1e-5 * np.abs(want).max()
    grad_sig = _view(nn, np.full(pred.shape, 7.0, np.float32), 1 - offset)
    for x, out, ref in ((d_x, grad_sig, want_sig), (None, grad_sig, want)):
        lib.uocr_seg_grad_ragged(d_gt.ptr, x.ptr if x is not None else None, out.ptr, d_ext.ptr, n, h, w, c, ws.ptr,
                                 nn.CP.stream())
        got = out.get()
        assert not got[~inside].any()
        assert np.abs(got - ref).max() <= 1e-5 * np.abs(ref).max()


@pytest.mark.gpu
def test_seg_loss_ragged_full_extents_match_stacked_loss(nn):
    """With every extent equal to the canvas, uocr_seg_loss_ragged gives uocr_seg_loss's loss and gradient."""
    import ctypes
    from univer_ocr_b200._lib import lib
    rng = np.random.default_rng(12)
    n, h, w, c = 4, 37, 45, 2
    pred = rng.uniform(0.01, 0.99, (n, h, w, c)).astype(np.float32)
    gt = (rng.uniform(size=pred.shape) < 0.3).astype(np.float32)
    need = ctypes.c_size_t(0)
    lib.uocr_seg_loss_workspace(n, c, ctypes.byref(need))
    d_pred, d_gt = nn.CP.copy(pred), nn.CP.copy(gt)
    out = {}
    for ragged in (False, True):
        ws = nn.DeviceArray(((need.value + 7) // 8,), 'float64')
        loss, grad = nn.DeviceArray.zeros((1,)), nn.DeviceArray.zeros(pred.shape)
        if ragged:
            lib.uocr_seg_loss_ragged(0, d_pred.ptr, d_gt.ptr, grad.ptr, loss.ptr, _dev_i32(nn, [[h, w]] * n).ptr, n, h,
                                     w, c, ws.ptr, nn.CP.stream())
        else:
            lib.uocr_seg_loss(0, d_pred.ptr, d_gt.ptr, grad.ptr, loss.ptr, n, h * w, c, ws.ptr, nn.CP.stream())
        out[ragged] = float(loss.get()[0]), grad.get()
    assert abs(out[True][0] - out[False][0]) <= 1e-6 * abs(out[False][0])
    assert np.abs(out[True][1] - out[False][1]).max() <= 1e-6 * np.abs(out[False][1]).max()


@pytest.mark.gpu
def test_softmax_ce_rows_matches_float64(nn):
    """uocr_softmax_ce_rows against NumPy float64 over the row ranges of a windowed batch (1 row, whole canvas rows, odd
    counts), with the valid-row count and with another denominator; rows outside the ranges (NaN there) are not read and
    get an exactly zero gradient.  With ranges covering every row and denom = batch it equals uocr_softmax_ce bit for
    bit."""
    from univer_ocr_b200._lib import lib
    rng = np.random.default_rng(13)
    widths, W, classes = np.array([1, 11, 4, 7, 2]), 11, 37
    n = len(widths)
    ranges = np.stack([np.arange(n) * W, np.arange(n) * W + widths], axis=1)
    logits = rng.normal(0, 3, (n * W, classes)).astype(np.float32)
    gt = np.zeros_like(logits)
    gt[np.arange(n * W), rng.integers(0, classes, n * W)] = 1
    valid = np.zeros(n * W, bool)
    for a, b in ranges:
        valid[a:b] = True
    logits[~valid], gt[~valid] = np.nan, np.nan
    x = np.where(valid[:, None], logits, 0).astype(np.float64)
    p = np.exp(x - x.max(axis=1, keepdims=True))
    p /= p.sum(axis=1, keepdims=True)
    g64 = np.where(valid[:, None], gt, 0).astype(np.float64)
    d_logits, d_gt, d_ranges = nn.CP.copy(logits), nn.CP.copy(gt), _dev_i32(nn, ranges)
    for denom in (float(widths.sum()), 100.0):
        loss, grad, ws = nn.DeviceArray.zeros((1,)), nn.DeviceArray.full(logits.shape, 7.0), nn.DeviceArray((n * W,))
        lib.uocr_softmax_ce_rows(d_logits.ptr, d_gt.ptr, grad.ptr, loss.ptr, d_ranges.ptr, n, n * W, classes, denom,
                                 ws.ptr, nn.CP.stream())
        want_loss = -(g64 * np.log(np.where(valid[:, None], p, 1))).sum() / denom
        want = np.where(valid[:, None], (p - g64) / denom, 0)
        got = grad.get()
        assert abs(float(loss.get()[0]) - want_loss) <= 1e-5 * abs(want_loss)
        assert not got[~valid].any()
        assert np.abs(got - want).max() <= 1e-5 * np.abs(want).max()
    # every row in a range: the stacked loss, bit for bit
    logits = rng.normal(0, 3, (n * W, classes)).astype(np.float32)
    d_logits = nn.CP.copy(logits)
    full = _dev_i32(nn, np.stack([np.arange(n) * W, np.arange(n) * W + W], axis=1))
    res = []
    for rows in (False, True):
        loss, grad, ws = nn.DeviceArray.zeros((1,)), nn.DeviceArray.zeros(logits.shape), nn.DeviceArray((n * W,))
        if rows:
            lib.uocr_softmax_ce_rows(d_logits.ptr, d_gt.ptr, grad.ptr, loss.ptr, full.ptr, n, n * W, classes,
                                     float(n * W), ws.ptr, nn.CP.stream())
        else:
            lib.uocr_softmax_ce(d_logits.ptr, d_gt.ptr, grad.ptr, loss.ptr, n * W, classes, ws.ptr, nn.CP.stream())
        res.append((loss.get(), grad.get()))
    assert np.array_equal(res[0][0], res[1][0], equal_nan=True)
    assert np.array_equal(res[0][1], res[1][1], equal_nan=True)


# per network: canvas (N, H, W) and the extents of its images
RAGGED_CASES = {
    'monochrome': np.array([[40, 52], [17, 23], [8, 9], [33, 40], [25, 52]]),
    'paragraph': np.array([[48, 64], [20, 36], [32, 16], [44, 60], [12, 24]]),
    'line': np.array([[48, 64], [16, 32], [32, 48], [48, 16], [16, 64], [32, 32]]),
    'char': np.array([[32, 96], [32, 40], [32, 8], [32, 61], [32, 77]]),
}


def _case(name, seed):
    """(ext, canvas, images, per-image targets) with each image's target on its own output shape."""
    from univer_ocr_b200 import my_model
    rng = np.random.default_rng(seed)
    ext = RAGGED_CASES[name]
    H, W = ext.max(axis=0)
    canvas = np.zeros((len(ext), H, W, 1), np.float32)
    images, targets = [], []
    model = my_model.MAKERS[name]((1, H, W, 1))
    for i, (h, w) in enumerate(ext):
        images.append(rng.uniform(0, 1, (1, h, w, 1)).astype(np.float32))
        canvas[i, :h, :w] = images[i]
        shape = model.get_output_shapes([(1, int(h), int(w), 1)])[0]
        if name == 'char':
            t = np.zeros(shape, np.float32)
            t[np.arange(shape[0]), rng.integers(0, shape[1], shape[0])] = 1
        else:
            t = (rng.uniform(size=shape) < 0.3).astype(np.float32)
        targets.append(t)
    return ext, canvas, images, targets


def _target_canvas(model, name, ext, targets):
    """The per-image targets on the output canvas of the batch (rows [i * W, i * W + w_i) for Char)."""
    H, W = ext.max(axis=0)
    shape = model.get_output_shapes([(len(ext), int(H), int(W), 1)])[0]
    y = np.zeros(shape, np.float32)
    for i, t in enumerate(targets):
        if name == 'char':
            y[i * W:i * W + t.shape[0]] = t
        else:
            y[i, :t.shape[1], :t.shape[2]] = t[0]
    return y


def _model(name, seed, optimizer=None, regularized=False):
    """A fresh network with the oracle's golden start weights (centred and scaled so that activations stay O(1): no
    saturated sigmoid, no 0 * log 0 in Char's softmax), the weights test_gpu_round2.py's TF32 tolerance is stated for.
    Without `regularized` the L2 regularisers are dropped: a sum over per-image steps would count them once per
    image."""
    from oracle import np_models
    from univer_ocr_b200 import my_model
    model = my_model.MAKERS[name]((1, 32, 32, 1), optimizer=optimizer)
    w = np_models.golden_weights(name, seed)
    model.set_weights({k: {n: v.tolist() for n, v in p.items()} for k, p in w.items()})
    if not regularized:
        for layer in model.layers.values():
            layer.regularizer = None
    return model


def _grads(model):
    return {k: p.grad.get().astype(np.float64) for k, p in model.params().items()}


def _rel_err(got, want):
    return max(np.abs(got[k] - want[k]).max() / max(np.abs(want[k]).max(), 1e-30) for k in want)


@pytest.mark.gpu
@pytest.mark.parametrize('mode', ['fp32', 'tf32'])
@pytest.mark.parametrize('name', ['monochrome', 'paragraph', 'line', 'char'])
def test_ragged_loss_and_gradients_equal_per_image_sums(nn, name, mode):
    """compute_loss_and_gradients_ragged over 5-6 images of different sizes == compute_loss_and_gradients on each image
    alone, summed (Dice) or weighted by w_i / sum(w) (Char).  FP32: the loss and every parameter gradient within 1e-4
    of the tensor's largest entry.  TF32, where shape-dependent kernel choices differ between the canvas and the single
    images: measured against the FP32 per-image result, the ragged step is within 2e-3 of each tensor's largest entry
    (the whole-network TF32 tolerance of test_gpu_round2.py) or at most three times as far off as the TF32 per-image
    steps themselves: weight gradients that cancel over many pixels (Char conv_1) carry about 1e-2 of TF32 rounding on
    either side."""
    ext, canvas, images, targets = _case(name, 20)
    model = _model(name, 21)
    total_w = float(ext[:, 1].sum())

    def per_image():
        loss, grads = 0.0, None
        for i, (X, t) in enumerate(zip(images, targets)):
            weight = ext[i, 1] / total_w if name == 'char' else 1.0
            out = model.compute_loss_and_gradients(nn.CP.copy(X), nn.CP.copy(t))
            loss += weight * float(out['output_losses'][0])
            g = _grads(model)
            grads = {k: weight * v for k, v in g.items()} if grads is None else {k: grads[k] + weight * g[k] for k in g}
        return loss, grads

    nn.CP.set_math_mode('fp32')
    want_loss, want = per_image()
    nn.CP.set_math_mode(mode)
    y = _target_canvas(model, name, ext, targets)
    out = model.compute_loss_and_gradients_ragged(nn.CP.copy(canvas), ext, nn.CP.copy(y))
    got_loss, got = float(out['output_losses'][0]), _grads(model)
    if mode == 'fp32':
        assert abs(got_loss - want_loss) <= 1e-4 * abs(want_loss), (name, got_loss, want_loss)
        for k in want:
            assert _rel_err({k: got[k]}, {k: want[k]}) <= 1e-4, (name, k)
        return
    tf_loss, tf = per_image()
    assert abs(got_loss - want_loss) <= max(2e-3 * abs(want_loss), 3 * abs(tf_loss - want_loss)), (name, got_loss)
    for k in want:
        err, ref = _rel_err({k: got[k]}, {k: want[k]}), _rel_err({k: tf[k]}, {k: want[k]})
        assert err <= max(2e-3, 3 * ref), (name, k, err, ref)


@pytest.mark.gpu
@pytest.mark.parametrize('mode', ['fp32', 'tf32'])
@pytest.mark.parametrize('name', ['monochrome', 'paragraph', 'line', 'char'])
def test_train_ragged_without_padding_is_the_stacked_step(nn, name, mode):
    """Every extent equal to the canvas: compute_loss_and_gradients_ragged == compute_loss_and_gradients (losses and
    gradients), train_ragged == train on the stacked batch (losses and updated weights over two steps), bit for bit,
    and the ragged step launches exactly the stacked step's kernels -- no mask.  Char's split-K weight gradients add
    their partial tiles with atomics, so its stacked step is not bit-reproducible against itself either.  There the
    gradients and the first step's loss agree within 1e-6 of their largest entry, and the weights after one step within
    1e-6 of each tensor's largest weight where the gradient is decided (|g| > 1e-3 max |g|), elsewhere within one Adam
    step (3.2 lr): Adam without bias correction moves a weight by ~3.2 lr sign(g) even for a gradient that rounding
    decides."""
    from univer_ocr_b200._lib import launch_count
    nn.CP.set_math_mode(mode)
    ext, canvas, images, targets = _case(name, 30)
    H, W = ext.max(axis=0)
    rng = np.random.default_rng(31)
    X = rng.uniform(0, 1, canvas.shape).astype(np.float32)
    full = np.tile([H, W], (len(ext), 1))
    lr = 1e-3
    a = _model(name, 32, optimizer=nn.optimizers.Adam(lr=lr))
    b = _model(name, 32, optimizer=nn.optimizers.Adam(lr=lr))
    shape = a.get_output_shapes([X.shape])[0]
    if name == 'char':
        y = np.zeros(shape, np.float32)
        y[np.arange(shape[0]), rng.integers(0, shape[1], shape[0])] = 1
    else:
        y = (rng.uniform(size=shape) < 0.3).astype(np.float32)
    tol = 1e-6 if name == 'char' else 0.0

    def same(u, v):
        u, v = np.asarray(u, np.float64), np.asarray(v, np.float64)
        return np.abs(u - v).max() <= tol * np.abs(u).max()

    dX, dy = nn.CP.copy(X), nn.CP.copy(y)
    la = float(a.compute_loss_and_gradients(dX, dy)['output_losses'][0])
    lb = float(b.compute_loss_and_gradients_ragged(dX, full, dy)['output_losses'][0])
    assert same([la], [lb]), (la, lb)
    ga, gb = _grads(a), _grads(b)
    for k in ga:
        assert same(ga[k], gb[k]), k
    for step in range(1 if name == 'char' else 2):
        n0 = launch_count()
        la = float(a.train(dX, dy)['output_losses'][0])
        n1 = launch_count()
        lb = float(b.train_ragged(dX, full, dy)['output_losses'][0])
        n2 = launch_count()
        assert same([la], [lb]), (step, la, lb)
        assert n2 - n1 == n1 - n0
    for (k, pa), pb in zip(a.params().items(), b.params().values()):
        u, v = pa.value.get().astype(np.float64), pb.value.get().astype(np.float64)
        decided = np.abs(ga[k]) > 1e-3 * np.abs(ga[k]).max()
        diff = np.abs(u - v)
        assert (diff[decided] <= tol * np.abs(u).max()).all(), k
        assert (diff <= (3.2 * lr if tol else 0.0)).all(), k


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['monochrome', 'char'])
def test_train_ragged_fused_equals_per_parameter_route(nn, name):
    """train_ragged's fused flat update == compute_loss_and_gradients_ragged + the per-parameter update (with the
    networks' own L2 regularisers), and test_ragged's loss == the training forward's loss (FP32)."""
    from univer_ocr_b200 import my_model
    nn.CP.set_math_mode('fp32')
    ext, canvas, images, targets = _case(name, 40)
    models = []
    for fused in (True, False):
        m = _model(name, 41, optimizer=nn.optimizers.Adam(lr=1e-3), regularized=True)
        m.fused_update = fused
        models.append(m)
    y = _target_canvas(models[0], name, ext, targets)
    dX, dy = nn.CP.copy(canvas), nn.CP.copy(y)
    test_loss = float(models[0].test_ragged(dX, ext, dy)['output_losses'][0])
    losses = [float(m.train_ragged(dX, ext, dy)['output_losses'][0]) for m in models]
    assert abs(losses[0] - losses[1]) <= 1e-6 * abs(losses[1])
    assert abs(test_loss - losses[0]) <= 1e-4 * abs(losses[0])
    for (k, pa), pb in zip(models[0].params().items(), models[1].params().values()):
        a, b = pa.value.get(), pb.value.get()
        assert np.abs(a - b).max() <= 1e-5 * np.abs(b).max(), k


class _CharLines:
    """Char samples: (1, 32, w, 1) line crops with w one-hot rows of labels."""

    def __init__(self, widths, seed):
        from univer_ocr_b200 import my_model
        rng = np.random.default_rng(seed)
        self.samples = []
        for w in widths:
            X = rng.uniform(0, 1, (1, 32, w, 1)).astype(np.float32)
            y = np.zeros((w, my_model.N_CHARS), np.float32)
            y[np.arange(w), rng.integers(0, my_model.N_CHARS, w)] = 1
            self.samples.append({'char': (X, y)})

    def __len__(self):
        return len(self.samples)

    def get(self, i):
        return self.samples[i]


@pytest.mark.gpu
def test_trainer_epoch_over_variable_size_lines(nn):
    """A Trainer epoch over line crops of different widths runs, and its one training step leaves the same weights as a
    hand-built DataParallel.train_ragged on the same canvas (within 1e-6 of each tensor's largest entry: Char's
    split-K weight gradients add partial tiles with atomics)."""
    from univer_ocr_b200 import my_model
    from univer_ocr_b200.parallel import DataParallel
    from univer_ocr_b200.trainer import Trainer
    nn.CP.set_math_mode('tf32')
    widths = [40, 97, 64, 23]
    train_ds, val_ds = _CharLines(widths, 50), _CharLines([30, 55, 55], 51)
    a = my_model.make_char((1, 32, 32, 1))
    b = my_model.make_char((1, 32, 32, 1))
    b.set_weights(a.get_weights())
    t = Trainer({'char': a}, train_ds, val_ds, batch_size=4, shuffle=lambda order: None, log=lambda *x, **k: None)
    best, _ = t.train(1)
    assert np.isfinite(best['char'][0])
    canvas = np.zeros((4, 32, max(widths), 1), np.float32)
    y = np.zeros((4 * max(widths), my_model.N_CHARS), np.float32)
    for i, w in enumerate(widths):
        X_i, y_i = train_ds.get(i)['char']
        canvas[i, :, :w] = X_i[0]
        y[i * max(widths):i * max(widths) + w] = y_i
    DataParallel(b).train_ragged(nn.CP.copy(canvas), np.array([[32, w] for w in widths]), nn.CP.copy(y))
    for (k, pa), pb in zip(a.params().items(), b.params().values()):     # split-K atomics: not bit-reproducible
        u, v = pa.value.get(), pb.value.get()
        assert np.abs(u - v).max() <= 1e-6 * np.abs(u).max(), k
