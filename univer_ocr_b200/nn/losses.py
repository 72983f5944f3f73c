"""Losses (reference: nn/losses.py).  `loss(prediction, ground_truth) -> (loss, grad)` as in
the reference; `loss` is a LazyScalar (behaves like the reference's float, but the device is
only synchronised when the number is actually read)."""
import ctypes

from .._lib import SEG_DICE, SEG_JACCARD, lib
from .gpu import DeviceArray, LazyScalar, as_device, stream


class BaseLoss:
    def __call__(self, prediction, ground_truth, want_grad=True):
        raise NotImplementedError()


class LazySegGrad:
    """The gradient of a Dice / Jaccard loss before it is written out: per-(n, c) coefficients a, b on the device
    (grad = a * gt + b, losses.py:24).  Handed to a `Sigmoid` layer's backward it becomes ONE pass that also applies
    the Sigmoid derivative (`uocr_seg_grad` with x_pre); anything else that touches it (`as_device`, `.get()`,
    arithmetic, attribute access) materialises the plain gradient tensor first."""

    def __init__(self, gt, workspace, shape):
        self._gt, self._ws, self.shape = gt, workspace, tuple(shape)
        self._dense = None

    def _dims(self):
        n, h, w, c = self.shape
        return n, h * w, c

    def _grad(self, x_pre_ptr, out_ptr):
        lib.uocr_seg_grad(self._gt.ptr, x_pre_ptr, out_ptr, *self._dims(), self._ws.ptr, stream())

    def materialize(self):
        if self._dense is None:
            out = DeviceArray(self.shape)
            self._grad(None, out.ptr)
            self._dense = out
        return self._dense

    def through_sigmoid(self, x_pre):
        """dL/dx for prediction = sigmoid(x_pre): (a * gt + b) * exp(-x) / (1 + exp(-x))^2 (layers.py:413-415)."""
        if self._dense is not None:
            return None
        dx = DeviceArray(self.shape)
        self._grad(x_pre.ptr, dx.ptr)
        return dx

    def __radd__(self, other):                              # Model.backward sums fan-out gradients: 0 + g
        if isinstance(other, (int, float)) and other == 0:
            return self
        return as_device(other) + self.materialize()

    def __add__(self, other):
        return self.materialize() + as_device(other)

    def __getattr__(self, name):                            # .get(), .ptr, .size, .reshape, ... of the dense tensor
        if name.startswith('_'):
            raise AttributeError(name)
        return getattr(self.materialize(), name)

    def __array__(self, dtype=None, copy=None):
        return self.materialize().__array__(dtype)


class LazySegGradRagged(LazySegGrad):
    """`LazySegGrad` of a ragged batch (`_Segmentation.ragged`): the gradient is written by uocr_seg_grad_ragged, so it
    is 0 outside each image's extent, with or without the Sigmoid derivative."""

    def __init__(self, gt, workspace, shape, extents, offset):
        super().__init__(gt, workspace, shape)
        self._ext, self._off = extents, offset

    def _grad(self, x_pre_ptr, out_ptr):
        lib.uocr_seg_grad_ragged(self._gt.ptr, x_pre_ptr, out_ptr, self._ext.ptr + 4 * self._off, *self.shape,
                                 self._ws.ptr, stream())


class _Segmentation(BaseLoss):
    kind = None

    def ragged(self, prediction, ground_truth, extents, offset=0, want_grad=True):
        """The loss of a ragged batch: (N, H, W, C) canvases, image n in its (h_n, w_n) region, the int32 (N, 2) table
        of those extents at `extents` (a device array) + `offset` int32 elements.  Sums over each region only; the
        loss is the sum of the per-image losses, as for a stacked batch."""
        pred, gt = as_device(prediction), as_device(ground_truth)
        assert pred.shape == gt.shape and pred.ndim == 4, f'{pred.shape} vs {gt.shape}'
        n, h, w, c = pred.shape
        need = ctypes.c_size_t(0)
        lib.uocr_seg_loss_workspace(n, c, ctypes.byref(need))
        ws = DeviceArray((need.value + 7) // 8, 'float64')
        loss = DeviceArray((1,))
        lib.uocr_seg_loss_ragged(self.kind, pred.ptr, gt.ptr, None, loss.ptr, extents.ptr + 4 * offset, n, h, w, c,
                                 ws.ptr, stream())
        return LazyScalar(loss), (LazySegGradRagged(gt, ws, pred.shape, extents, offset) if want_grad else None)

    def __call__(self, prediction, ground_truth, want_grad=True):
        pred, gt = as_device(prediction), as_device(ground_truth)
        assert pred.shape == gt.shape, f'{pred.shape} != {gt.shape}'
        n, h, w, c = pred.shape
        need = ctypes.c_size_t(0)
        lib.uocr_seg_loss_workspace(n, c, ctypes.byref(need))
        ws = DeviceArray((need.value + 7) // 8, 'float64')
        loss = DeviceArray((1,))
        lib.uocr_seg_loss(self.kind, pred.ptr, gt.ptr, None, loss.ptr, n, h * w, c, ws.ptr, stream())
        return LazyScalar(loss), (LazySegGrad(gt, ws, pred.shape) if want_grad else None)


class SegmentationDice2D(_Segmentation):
    """losses.py:9-25"""
    kind = SEG_DICE


class SegmentationJaccard2D(_Segmentation):
    """losses.py:28-42"""
    kind = SEG_JACCARD


class SigmoidCrossEntropy(BaseLoss):
    """losses.py:45-57"""

    def __call__(self, prediction, ground_truth, want_grad=True):
        pred, gt = as_device(prediction), as_device(ground_truth)
        assert pred.shape == gt.shape, f'{pred.shape} != {gt.shape}'
        batch = gt.shape[0]
        loss = DeviceArray((1,))
        grad = DeviceArray(pred.shape) if want_grad else None
        lib.uocr_sigmoid_ce(pred.ptr, gt.ptr, grad.ptr if want_grad else None, loss.ptr, batch,
                            pred.size // batch, stream())
        return LazyScalar(loss), grad


class SoftmaxCrossEntropy(BaseLoss):
    """losses.py:60-73"""

    def __call__(self, prediction, ground_truth, want_grad=True):
        pred, gt = as_device(prediction), as_device(ground_truth)
        assert pred.shape == gt.shape and pred.ndim == 2, f'{pred.shape} vs {gt.shape}'
        batch, classes = pred.shape
        loss = DeviceArray((1,))
        ws = DeviceArray((batch,))
        grad = DeviceArray(pred.shape) if want_grad else None
        lib.uocr_softmax_ce(pred.ptr, gt.ptr, grad.ptr if want_grad else None, loss.ptr, batch,
                            classes, ws.ptr, stream())
        return LazyScalar(loss), grad

    def rows(self, prediction, ground_truth, ranges, offset, n_ranges, denom, want_grad=True):
        """The loss over the rows of a windowed ragged batch: the int32 (n_ranges, 2) [first, end) table at `ranges` (a
        device array) + `offset` int32 elements.  loss = -sum(gt * log p) over those rows / denom; every other row adds
        nothing and gets a zero gradient."""
        pred, gt = as_device(prediction), as_device(ground_truth)
        assert pred.shape == gt.shape and pred.ndim == 2, f'{pred.shape} vs {gt.shape}'
        batch, classes = pred.shape
        loss = DeviceArray((1,))
        ws = DeviceArray((batch,))
        grad = DeviceArray(pred.shape) if want_grad else None
        lib.uocr_softmax_ce_rows(pred.ptr, gt.ptr, grad.ptr if want_grad else None, loss.ptr,
                                 ranges.ptr + 4 * offset, n_ranges, batch, classes, float(denom), ws.ptr, stream())
        return LazyScalar(loss), grad
