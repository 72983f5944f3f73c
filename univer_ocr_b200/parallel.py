"""Batch-sharded data-parallel training step (SURVEY.md 8e).

One process per GPU; every rank runs the step on its shard of the batch:

    forward + loss + backward     gradients accumulate into the model's flat gradient buffer (nn/flat.py)
      |  while backward runs: as soon as a layer's parameter gradients are final, the contiguous flat range they
      |  complete is sum-allreduced over NVLink / NVSwitch on the communicator's SIDE stream (buckets grow in
      |  reverse layer order, so the Char head's FullyConnected gradients -- 99 % of my_model's 3.2 MB -- are on
      |  the wire while the convolutions' backward is still computing)
    join: the compute stream waits for the last bucket
    ONE fused kernel per regularisation group: g*scale + 2*l2*w -> Adam -> w   (+ reg loss)
    ONE memset of the flat gradient buffer

The collectives go through libuocr's own NCCL binding (`comm.Communicator` over `uocr_allreduce_sum_f32`); no
PyTorch anywhere.  The whole step -- collectives included -- is a fixed launch sequence over fixed buffers and
can be replayed from one CUDA graph (`pipeline.CapturedStep`).

Gradient scaling: the Dice / Jaccard losses sum over the batch (`losses.py:23`), so shard gradients are summed
without scaling; SoftmaxCE / SigmoidCE divide by the LOCAL batch (`losses.py:69-72`), so their summed gradients are
scaled by 1 / world (= local / global batch).  A ragged SoftmaxCE step (`train_ragged` with `rows_total`) divides by
the valid rows of all ranks instead and is not scaled.  The L2 gradient depends on the weights only, so it is added once,
after the allreduce (inside the fused update).
"""
import ctypes

from . import comm as comm_
from ._lib import lib
from .nn import optimizers
from .nn.flat import BucketScheduler, FlatParameters          # noqa: F401  (FlatParameters: public name)
from .nn.gpu import CP, LazyScalar
from .nn.losses import SegmentationDice2D, SegmentationJaccard2D


def _new_event():
    e = ctypes.c_void_p()
    lib.uocr_event_create(ctypes.byref(e))
    return e.value


class DataParallel:
    """One training step of `model` on this rank's shard of the batch.

        comm.init_from_env()                        # once per process (torchrun's RANK / WORLD_SIZE / LOCAL_RANK)
        dp = DataParallel(model, optimizer)
        losses = dp.train(X_shard, y_shard)         # same dict as Model.train

    With world == 1 this is simply the fused single-GPU step (what `Model.train` itself runs).
    `overlap=False` issues ONE allreduce over the whole flat buffer after backward, on the compute stream."""

    def __init__(self, model, optimizer=None, comm=None, overlap=True, bucket_bytes=256 << 10):
        self.model = model
        self.optimizer = optimizer if optimizer is not None else self._find_optimizer(model)
        if not isinstance(self.optimizer, optimizers.Adam):
            raise NotImplementedError('DataParallel fuses the Adam update (the only optimiser my_model uses)')
        self.flat = model.flat_parameters()
        if self.flat is None or model.fused_optimizer() is not self.optimizer:
            raise NotImplementedError('DataParallel needs a model whose parameters share this Adam instance, '
                                      'regularised by L2 or nothing (nn.flat.FlatParameters.eligible)')
        self.comm = comm if comm is not None else comm_.current()
        self.world, self.rank = self.comm.world, self.comm.rank
        self.overlap = bool(overlap) and self.world > 1
        self.scheduler = BucketScheduler(self.flat.layer_ranges, max(1, int(bucket_bytes) // 4))
        self._ev_ready, self._ev_joined = (_new_event(), _new_event()) if self.world > 1 else (None, None)
        self.buckets_last_step = []                     # [(lo, hi)] of the last step, in issue order
        self.after_reduce = None                        # optional callable: sees the summed gradients before the update
        losses = model.loss if isinstance(model.loss, list) else [model.loss]
        summed = all(isinstance(l, (SegmentationDice2D, SegmentationJaccard2D)) for l in losses)
        self.grad_scale = 1.0 if summed else 1.0 / self.world
        if self.world > 1:
            self.broadcast_parameters()

    @staticmethod
    def _find_optimizer(model):
        for layer in model.layers.values():
            for param in layer.params().values():
                return param.optimizer
        raise ValueError('model has no parameters')

    def broadcast_parameters(self, src=0):
        """Rank `src`'s parameters (and Adam state) on every rank."""
        st = CP.stream()
        for buf in (self.flat.values, self.flat.velocity, self.flat.accumulated):
            self.comm.broadcast(buf, src, stream=st)
        CP.weights_generation += 1

    # ---- gradient reduction -----------------------------------------------------------
    def _send(self, lo, hi):
        """Sum-allreduce flat.grads[lo:hi] on the communicator's stream, after everything queued so far on the
        current compute stream (the kernels that produced those gradients)."""
        side = self.comm.stream
        lib.uocr_event_record(self._ev_ready, CP.stream())
        lib.uocr_stream_wait_event(side, self._ev_ready)
        self.comm.allreduce_sum(self.flat.grads, lo, hi - lo, stream=side)
        self.buckets_last_step.append((lo, hi))

    def _layer_done(self, name):
        for lo, hi in self.scheduler.layer_done(name):
            self._send(lo, hi)

    def allreduce_gradients(self):
        """After backward: flush what the buckets still hold and make the compute stream wait for the wire."""
        if self.world == 1:
            return
        if not self.overlap:
            self.comm.allreduce_sum(self.flat.grads, stream=CP.stream())
            self.buckets_last_step = [(0, self.flat.total)]
            return
        for lo, hi in self.scheduler.finish():
            self._send(lo, hi)
        lib.uocr_event_record(self._ev_joined, self.comm.stream)
        lib.uocr_stream_wait_event(CP.stream(), self._ev_joined)

    def _reduce(self):
        self.allreduce_gradients()
        if self.after_reduce is not None:
            self.after_reduce()

    def update(self):
        """Fused L2 + Adam over the flat buffers, then zero the gradients -> regularisation loss."""
        reg = self.flat.update(self.optimizer, self.grad_scale)
        return reg if isinstance(reg, LazyScalar) else LazyScalar(_zero_scalar())

    def train(self, X, y):
        self.scheduler.reset()
        self.buckets_last_step = []
        hook = self._layer_done if self.overlap else None
        out = self.model.train_fused(X, y, reduce_gradients=self._reduce, grad_scale=self.grad_scale,
                                     on_layer_done=hook)
        return self._finish(out)

    def train_ragged(self, canvas, extents, y, rows_total=None):
        """`train` on this rank's ragged batch (Model.train_fused_ragged).  Dice / Jaccard losses sum over images, so
        the summed gradients are the global ones.  A mean-over-rows loss given `rows_total`, the valid rows of all
        ranks, is already divided by the global count, so its summed gradients are not scaled either; without it the
        1 / world rule of `train` applies."""
        self.scheduler.reset()
        self.buckets_last_step = []
        hook = self._layer_done if self.overlap else None
        scale = 1.0 if rows_total is not None else self.grad_scale
        out = self.model.train_fused_ragged(canvas, extents, y, rows_total=rows_total, reduce_gradients=self._reduce,
                                            grad_scale=scale, on_layer_done=hook)
        return self._finish(out)

    @staticmethod
    def _finish(out):
        if not isinstance(out['regularization_loss'], LazyScalar):
            out['regularization_loss'] = LazyScalar(_zero_scalar())
        return out


def _zero_scalar():
    from .nn.gpu import DeviceArray
    return DeviceArray.zeros((1,))
