"""Batched, data-parallel epoch driver for the four sub-networks (SURVEY.md 8f, row 1).

Mirrors `my_model/trainer.py` of the reference (`Losses` :10-128, `Trainer` :131-296): losses of
the validation set are computed before the first epoch; every epoch shuffles the training order,
then the validation order, trains, validates, normalises the accumulated losses by the data set
sizes, decays the learning rate by `learning_rate_step ** reload_attempts`, rolls the weights back
when a NaN shows up in any model (last epoch's weights for the first 9 attempts in a row, then
the weights the run started from, with the attempt counter reset -- the reference never refreshes
its `best_weights` after the start, `trainer.py:185`, and neither does this class), reports which
models improved on their best validation loss to `save_weights_func`, and returns
`(val_best_losses, best_loss_epoch)`.

What is different, on purpose:

* the reference feeds ONE sample per step through its `model_system` (crop / rotate glue on the
  host between the networks, out of scope here) and calls `gc.collect()` after each
  (`trainer.py:231-232`).  Here every model gets its own batches: a data set's `get(i)` returns
  `{model_name: (X, y)}` with a leading batch axis, `batch_size` of them are stacked per step and,
  with a multi-rank communicator (`univer_ocr_b200.comm`, NCCL through libuocr -- no PyTorch), each rank trains
  its slice of the stack through `parallel.DataParallel` (bucketed NCCL allreduce of the flat gradient buffer,
  overlapped with backward); rank 0's shuffled orders are broadcast so that the ranks' slices partition each
  batch, and at world > 1 every sample must carry every model (a rank that skipped a model's step would leave
  the others waiting in that model's allreduce);
* loss values stay on the device during an epoch (`LazyScalar`), the epoch's sums are read back
  once and summed over ranks, so every rank takes the same NaN / best-weights decisions;
* roll-back snapshots of `Model`s are device copies of the flat parameter buffer (3.2 MB) instead
  of `get_weights()` nested lists (the reference's 16.5 MB of Python floats per epoch).

Losses that average over the local batch (SoftmaxCE / SigmoidCE, `nn/losses.py:69-72`) are
weighted by the number of stacked samples so that an epoch's sum equals the reference's sum of
per-sample losses (exactly for equal sample sizes); Dice / Jaccard already sum over the batch.

Samples of different sizes -- the reference's data: pages, paragraph crops and line crops differ in
size -- are batched too.  When a model's samples in a batch differ in any axis but the first, they
are packed on the host instead of stacked: X on a zero-filled (N, H, W, C) canvas with each image's
(h, w) in a table of extents, y on its output canvas (image maps) or in its row ranges (window
rows), and the batch runs through `train_ragged` / `test_ragged` (`Model.train_ragged`, DESIGN.md
§3).  At world > 1 a mean-over-batch model's training step sums [ragged?, valid rows, samples] over
the ranks with one `allreduce_host`, so that every rank takes the same path; a ragged step then
divides its loss by the valid rows of all ranks and is weighted by the samples of all ranks.

Any object with `train(X, y) / test(X, y) / get_weights() / set_weights(w) / nan_weights() /
get_outputs_count()` is accepted as a model (used as is); `nn.models.Model` instances are wrapped
in `DataParallel` unless `fused_update=False`.
"""
import random
from datetime import datetime as dt

import numpy as np


class Losses:
    """Per-model, per-output loss bookkeeping of one run (`my_model/trainer.py:10-57`)."""

    def __init__(self, model_names, outputs_cnts):
        self.model_names = model_names
        self.outputs_cnts = outputs_cnts
        self.train_prev_losses = self._new_losses(float('inf'))
        self.val_best_losses = self._new_losses(float('inf'))
        self.val_prev_losses = self._new_losses(float('inf'))
        self.train_losses = None
        self.val_losses = None
        self.best_loss_epoch = {name: 0 for name in self.model_names}
        self._pending = []

    def _new_losses(self, value):
        return {name: [value] * self.outputs_cnts[name] for name in self.model_names}

    def reset(self):
        self.train_losses = self._new_losses(0)
        self.val_losses = self._new_losses(0)
        self._pending = []

    def next(self):
        self.train_prev_losses = self.train_losses
        self.val_prev_losses = self.val_losses

    def _add(self, target, update, weight=1):
        for name in self.model_names:
            if name not in update:
                continue
            out_losses = update[name]['output_losses']
            for i in range(self.outputs_cnts[name]):
                if isinstance(out_losses[i], (int, float)):
                    target[name][i] = target[name][i] + out_losses[i] * weight
                else:                                    # device-resident value: no read-back (= sync) per step
                    self._pending.append((target, name, i, out_losses[i], weight))

    def train(self, update, weight=1):
        self._add(self.train_losses, update, weight)

    def validation(self, update, weight=1):
        self._add(self.val_losses, update, weight)

    def materialize(self, reduce_fn=None):
        """Adds the device-resident values of the epoch (read back here, in step order) and, with `reduce_fn`,
        sums the tables over ranks."""
        for target, name, i, loss, weight in self._pending:
            target[name][i] = target[name][i] + float(loss) * weight
        self._pending = []
        flat = [float(v) for table in (self.train_losses, self.val_losses)
                for name in self.model_names for v in table[name]]
        if reduce_fn is not None:
            flat = reduce_fn(flat)
        it = iter(flat)
        for table in (self.train_losses, self.val_losses):
            for name in self.model_names:
                table[name] = [next(it) for _ in range(self.outputs_cnts[name])]

    def normalize(self, train_dataset_size, validation_dataset_size):
        for name in self.model_names:
            for i in range(self.outputs_cnts[name]):
                self.train_losses[name][i] /= train_dataset_size
                self.val_losses[name][i] /= validation_dataset_size

    def get_better_weights(self, epoch):
        """Names of the models whose mean validation loss improved (a finite loss also beats a
        NaN best), `trainer.py:31-41`."""
        def better(a, b):
            return bool(np.mean(a) < np.mean(b)) or (not np.any(np.isnan(a)) and bool(np.any(np.isnan(b))))
        result = [name for name in self.model_names
                  if better(self.val_losses[name], self.val_best_losses[name])]
        for name in result:
            self.val_best_losses[name] = self.val_losses[name]
            self.best_loss_epoch[name] = epoch
        return result

    def print(self, left_margin=0, out=print):
        """The reference's table (`trainer.py:59-128`): values, change against the previous epoch,
        mean change, for training and validation."""
        def fmt(table, prev):
            values = [[f'{v: }' for v in table[n]] for n in self.model_names]
            diffs = [[table[n][i] - prev[n][i] for i in range(self.outputs_cnts[n])] for n in self.model_names]
            return values, [[f'{d:+}' for d in row] for row in diffs], [f'{np.mean(row):+}' for row in diffs]
        t_val, t_diff, t_avg = fmt(self.train_losses, self.train_prev_losses)
        v_val, v_diff, v_avg = fmt(self.val_losses, self.val_prev_losses)
        widths = []
        for m, name in enumerate(self.model_names):
            cols = [max(len(rows[m][j]) for rows in (t_val, v_val, t_diff, v_diff))
                    for j in range(self.outputs_cnts[name])]
            for rows in (t_val, v_val, t_diff, v_diff):
                rows[m] = ' '.join(cell.ljust(cols[j]) for j, cell in enumerate(rows[m]))
            widths.append(max(len(name), sum(cols), len(t_avg[m]), len(v_avg[m])))
        lm = ' ' * left_margin
        labels = ['Models:            ', 'Train loss:        ', '  Loss change:     ', '  Avg loss change: ',
                  'Validation loss:   ', '  Loss change:     ', '  Avg loss change: ']
        for label, row in zip(labels, (list(self.model_names), t_val, t_diff, t_avg, v_val, v_diff, v_avg)):
            out(lm + label + ' | '.join(cell.ljust(widths[m]) for m, cell in enumerate(row)))


def _mean_over_batch(model):
    """True when the model's losses divide by the local batch (SoftmaxCE / SigmoidCE)."""
    try:
        from .nn.losses import SegmentationDice2D, SegmentationJaccard2D
    except Exception:                                   # noqa: BLE001 -- duck-typed models only
        return False
    loss = getattr(model, 'loss', None)
    if loss is None:
        return False
    losses = loss if isinstance(loss, list) else [loss]
    return not all(isinstance(l, (SegmentationDice2D, SegmentationJaccard2D)) for l in losses)


class _Stepper:
    """One model behind the trainer: how to step it, snapshot it and roll it back."""

    def __init__(self, model, optimizer, fused_update, comm=None):
        self.model, self.dp = model, None
        is_native = False
        try:
            from .nn.models import Model
            is_native = isinstance(model, Model)
        except Exception:                               # noqa: BLE001 -- no CUDA library: fakes only
            pass
        self.mean_loss = _mean_over_batch(model) if is_native else bool(getattr(model, 'mean_over_batch', False))
        if is_native and fused_update:
            from .parallel import DataParallel
            self.dp = DataParallel(model, optimizer, comm=comm)

    def train(self, X, y):
        return (self.dp or self.model).train(X, y)

    def test(self, X, y):
        return self.model.test(X, y)

    def train_ragged(self, canvas, extents, y, rows_total=None):
        return (self.dp or self.model).train_ragged(canvas, extents, y, rows_total=rows_total)

    def test_ragged(self, canvas, extents, y):
        return self.model.test_ragged(canvas, extents, y)

    def snapshot(self):
        if self.dp is None:
            return self.model.get_weights()
        return self.dp.flat.snapshot()

    def restore(self, snapshot):
        if self.dp is None:
            self.model.set_weights(snapshot)
            return
        self.dp.flat.restore(snapshot)


class Trainer:
    """
        trainer = Trainer(models, train_dataset, validation_dataset, optimizer=adam,
                          learning_rate_step=0.995, batch_size=64, save_weights_func=save)
        best_losses, best_epochs = trainer.train(num_epochs=100)

    `models`: {name: model}.  Data sets: `len(ds)` samples, `ds.get(i)` → {name: (X, y)} where X / y
    are arrays (or lists of arrays for multi-input / multi-output models) with a leading batch
    axis; a model missing from the dict sits that sample out; the next `prefetch` batches are
    fetched and stacked by a background thread.  Stacking 64 page tiles on the host still costs
    ~20 ms, twenty times the GPU's training step, so a data set may instead offer
    `ds.get_batch(indices)` → {name: (X, y)} already stacked -- host or device arrays
    (`tools/train_synthetic.py` keeps its samples in HBM and gathers with device copies).  `save_weights_func(names)` is called
    on rank 0 with the models whose validation loss improved (`my_model/train.py:132-141`)."""

    MAX_RELOAD_ATTEMPTS = 10                            # trainer.py:262

    def __init__(self, models, train_dataset, validation_dataset, progress_tracker=None,
                 optimizer=None, learning_rate_step=0.995, save_weights_func=None,
                 batch_size=1, fused_update=True, shuffle=None, log=print, prefetch=2, comm=None):
        self.models = models
        self.train_dataset = train_dataset
        self.validation_dataset = validation_dataset
        self.progress_tracker = progress_tracker
        self.optimizer = optimizer
        self.learning_rate_step = learning_rate_step
        self.save_weights_func = save_weights_func
        self.batch_size = int(batch_size)
        self.shuffle = shuffle if shuffle is not None else random.shuffle   # trainer.py:3
        self.log = log
        self.prefetch = int(prefetch)
        if comm is None:
            from . import comm as comm_
            comm = comm_.current()
        self.comm = comm                                # rank / world / allreduce_host / broadcast_ints
        self.world, self.rank = comm.world, comm.rank
        assert self.batch_size % self.world == 0, (
            f'batch_size {self.batch_size} must be divisible by the world size {self.world}')
        assert min(len(train_dataset), len(validation_dataset)) >= self.world, 'fewer samples than ranks'
        self.steppers = {name: _Stepper(model, optimizer, fused_update, comm) for name, model in models.items()}

    # ---- plumbing -------------------------------------------------------------------
    def _message(self, *args):
        if self.progress_tracker is not None:
            self.progress_tracker.message(*args)

    def _reduce(self, values):
        return values if self.world == 1 else self.comm.allreduce_host(values, 'sum')

    def _shuffle(self, order):
        """The reference's in-place `random.shuffle` (`trainer.py:207,211`); with several ranks, rank 0's permutation
        is the epoch's order everywhere -- per-process shuffles would make the ranks' [rank::world] slices overlap."""
        self.shuffle(order)
        if self.world > 1:
            order[:] = self.comm.broadcast_ints(order, root=0)

    @staticmethod
    def _stack(parts):
        """[(X, y), ...] → (X, y) concatenated along the batch axis (lists element-wise)."""
        def cat(items):
            if isinstance(items[0], (list, tuple)):
                return [cat([it[k] for it in items]) for k in range(len(items[0]))]
            return items[0] if len(items) == 1 else np.concatenate(items, axis=0)
        return cat([p[0] for p in parts]), cat([p[1] for p in parts])

    @staticmethod
    def _ragged(parts):
        """True when the parts' X are image batches that differ in an axis other than the first (cannot be stacked)."""
        xs = [p[0] for p in parts]
        if any(isinstance(x, (list, tuple)) or np.ndim(x) != 4 for x in xs):
            return False
        return len({tuple(np.shape(x)[1:]) for x in xs}) > 1

    @staticmethod
    def _pack(parts):
        """[(X, y), ...] with X (k, h, w, C) of different sizes -> (canvas, extents, y, valid rows): X on a zero-filled
        (N, H, W, C) canvas, (H, W) the largest extents, a part with k images adding k rows (h, w) to the table.  A
        target that is an image map, (k, h', w', C'), goes on its zero-filled canvas the same way; one of window rows,
        (k * r, classes), puts image j's r rows at [j * R, j * R + r), R the largest r -- the layout of
        Model.ragged_train_analysis, since a network's output extents grow with its input's.  Valid rows: the rows of
        the first target (0 for image maps)."""
        xs = [np.asarray(p[0]) for p in parts]
        counts = [x.shape[0] for x in xs]
        n = sum(counts)
        canvas = np.zeros((n, max(x.shape[1] for x in xs), max(x.shape[2] for x in xs), xs[0].shape[3]), np.float32)
        ext = np.zeros((n, 2), np.int64)
        i = 0
        for x in xs:
            canvas[i:i + x.shape[0], :x.shape[1], :x.shape[2]] = x
            ext[i:i + x.shape[0]] = x.shape[1:3]
            i += x.shape[0]

        def place(items):
            if isinstance(items[0], (list, tuple)):
                return [place([it[k] for it in items]) for k in range(len(items[0]))]
            ts = [np.asarray(t) for t in items]
            if ts[0].ndim == 4:
                out = np.zeros((n, max(t.shape[1] for t in ts), max(t.shape[2] for t in ts), ts[0].shape[3]), np.float32)
                j = 0
                for t in ts:
                    out[j:j + t.shape[0], :t.shape[1], :t.shape[2]] = t
                    j += t.shape[0]
                return out
            per = [t.shape[0] // k for t, k in zip(ts, counts)]
            rows = max(per)
            out = np.zeros((n * rows, *ts[0].shape[1:]), np.float32)
            j = 0
            for t, k, r in zip(ts, counts, per):
                for m in range(k):
                    out[(j + m) * rows:(j + m) * rows + r] = t[m * r:(m + 1) * r]
                j += k
            return out

        y = place([p[1] for p in parts])
        first = [np.asarray(p[1][0] if isinstance(p[1], (list, tuple)) else p[1]) for p in parts]
        valid = sum(t.shape[0] for t in first) if first[0].ndim == 2 else 0
        return canvas, ext, y, valid

    def _batches(self, dataset, order):
        """`_host_batches` with the next `prefetch` batches fetched and stacked by a background thread while the
        current one trains (host data sets only: `get_batch` data sets do their own staging)."""
        source = self._host_batches(dataset, order)
        if self.prefetch <= 0 or hasattr(dataset, 'get_batch') or len(order) <= self.batch_size:
            yield from source
            return
        import queue
        import threading
        ready, stop, end = queue.Queue(maxsize=self.prefetch), threading.Event(), object()

        def produce():
            try:
                for item in source:
                    while not stop.is_set():
                        try:
                            ready.put(item, timeout=0.1)
                            break
                        except queue.Full:
                            continue
                    if stop.is_set():
                        return
                ready.put(end)
            except BaseException as exc:                 # noqa: BLE001 -- re-raised in the consumer
                ready.put(exc)

        worker = threading.Thread(target=produce, name='uocr-trainer-prefetch', daemon=True)
        worker.start()
        try:
            while True:
                item = ready.get()
                if item is end:
                    return
                if isinstance(item, BaseException):
                    raise item
                yield item
        finally:
            stop.set()

    def _host_batches(self, dataset, order):
        """Yields ({name: (X, y, n_samples, ragged)}, samples consumed so far): `batch_size` samples per
        step, this rank's share [rank::world] of each.  `ragged` is None for a stacked batch, else (extents, valid
        rows) of a packed one (X, y its canvases, `_pack`)."""
        batched = getattr(dataset, 'get_batch', None)
        for start in range(0, len(order), self.batch_size):
            chunk = order[start:start + self.batch_size]
            if self.world > 1 and len(chunk) % self.world:
                # every rank must take part in every step (the gradient allreduce is a collective): the last, ragged
                # stack keeps a multiple of the world size; `_usable` is what the epoch's losses are normalised by
                chunk = chunk[:len(chunk) - len(chunk) % self.world]
                if not chunk:
                    return
            mine = chunk[self.rank::self.world]
            if batched is not None:
                # the data set stacks (and may keep its samples on the device): {name: (X, y)} for these indices
                got = batched(mine)
                yield ({name: (X, y, len(mine), None) for name, (X, y) in got.items() if name in self.models},
                   start + len(chunk))
                continue
            samples = [dataset.get(i) for i in mine]
            batch = {}
            for name in self.models:
                parts = [s[name] for s in samples if name in s]
                if self.world > 1 and len(parts) != len(samples):
                    raise ValueError(f'data-parallel training needs every model in every sample: {name!r} is missing '
                                     f'from {len(samples) - len(parts)} of this rank\'s {len(samples)} samples (a rank '
                                     f'that skips a model\'s step leaves the others waiting in its allreduce)')
                if parts and self._ragged(parts):
                    X, ext, y, valid = self._pack(parts)
                    batch[name] = (X, y, len(parts), (ext, valid))
                elif parts:
                    X, y = self._stack(parts)
                    batch[name] = (X, y, len(parts), None)
            yield batch, start + len(chunk)

    def _run(self, dataset, order, training, losses):
        total = len(order)
        for batch, done in self._batches(dataset, order):
            if self.progress_tracker is not None:
                self.progress_tracker.reset()
            self._message('training' if training else 'validating')
            update, weights = {}, {}
            agree = training and self.world > 1 and not hasattr(dataset, 'get_batch')
            for name, (X, y, n, ragged) in batch.items():
                st = self.steppers[name]
                weights[name] = n if st.mean_loss else 1
                if agree and st.mean_loss:
                    update[name], weights[name] = self._train_mean_step(st, X, y, n, ragged)
                elif ragged is not None:
                    ext = ragged[0]
                    update[name] = st.train_ragged(X, ext, y) if training else st.test_ragged(X, ext, y)
                else:
                    update[name] = st.train(X, y) if training else st.test(X, y)
            for name in update:                          # one weight per model
                (losses.train if training else losses.validation)({name: update[name]}, weights[name])
            self._message('train_iteration' if training else 'val_iteration', {'current': done, 'total': total})

    def _train_mean_step(self, st, X, y, n, ragged):
        """A mean-over-batch model's training step at world > 1 -> (losses, weight).  The ranks sum [ragged?, valid rows,
        samples]; if any rank's batch is ragged, every rank takes the ragged step (a stacked batch is a canvas without
        padding) with the loss over the valid rows of all ranks, weighted by the samples of all ranks."""
        if ragged is not None:
            rows = ragged[1]
        else:
            first = y[0] if isinstance(y, (list, tuple)) else y
            rows = np.shape(first)[0] if np.ndim(first) == 2 else 0
        any_ragged, rows_total, samples = self.comm.allreduce_host([float(ragged is not None), float(rows), float(n)],
                                                                   'sum')
        if not any_ragged:
            return st.train(X, y), n
        ext = ragged[0] if ragged is not None else np.tile(np.shape(X)[1:3], (np.shape(X)[0], 1))
        return st.train_ragged(X, ext, y, rows_total=int(round(rows_total))), int(round(samples))

    def _usable(self, n):
        """Samples of an n-sample data set that a pass consumes (all of them on one rank)."""
        if self.world == 1:
            return n
        full, rest = divmod(n, self.batch_size)
        return full * self.batch_size + rest - rest % self.world

    def _nan_weights(self):
        return any(model.nan_weights() for model in self.models.values())

    # ---- the run --------------------------------------------------------------------
    def train(self, num_epochs):
        names = list(self.models.keys())
        losses = Losses(names, {name: m.get_outputs_count() for name, m in self.models.items()})
        log = self.log if self.rank == 0 else (lambda *a, **k: None)
        n_train, n_val = len(self.train_dataset), len(self.validation_dataset)

        log('Precomputing losses')
        ts = dt.now()
        losses.reset()
        self._run(self.validation_dataset, list(range(n_val)), False, losses)
        losses.materialize(self._reduce)
        losses.print(left_margin=2, out=log)
        losses.next()
        log(f'Time required: {dt.now() - ts}')
        log('\n')

        best = last = {name: st.snapshot() for name, st in self.steppers.items()}
        reload_attempts = 0
        train_order, val_order = list(range(n_train)), list(range(n_val))

        epoch = 1
        while epoch <= num_epochs:
            log(f'[{dt.now()}]')
            log(f'Epoch {str(epoch).rjust(len(str(num_epochs)))}/{num_epochs}:')
            self._message('epoch', {'current': epoch, 'total': num_epochs})
            self._message('train_iteration', {'current': 0, 'total': n_train})
            self._message('val_iteration', {'current': 0, 'total': n_val})
            if self.optimizer is not None:
                log(f'  lr = {self.optimizer.lr}')
            ts = dt.now()
            losses.reset()

            self._shuffle(train_order)
            self._run(self.train_dataset, train_order, True, losses)
            self._shuffle(val_order)
            assert n_val > 0, 'Validation dataset must have at least 1 element'
            self._run(self.validation_dataset, val_order, False, losses)
            losses.materialize(self._reduce)
            losses.normalize(self._usable(n_train), self._usable(n_val))

            if self.optimizer is not None:
                reload_attempts += 1
                self.optimizer.lr *= self.learning_rate_step ** reload_attempts
                if self._nan_weights():
                    if reload_attempts < self.MAX_RELOAD_ATTEMPTS:
                        log('NaN value found in weights, loading last weights\n')
                        source = last
                    else:
                        log('Too many attempts, loading last best weights\n')
                        source = best
                        reload_attempts = 0
                    for name, st in self.steppers.items():
                        st.restore(source[name])
                    continue
            elif self._nan_weights():
                raise ValueError(
                    'NaN value found in weights, but no optimizer provided. '
                    'Provide optimizer and learning_rate_step, so '
                    'learning rate could be decreased to try avoiding NaN values')

            losses.print(left_margin=2, out=log)
            better = losses.get_better_weights(epoch)
            if any(better) and self.save_weights_func and self.rank == 0:
                log('  Saving weights for ' + ', '.join(better))
                self.save_weights_func(better)
            log(f'Time required: {dt.now() - ts}')
            log('\n')

            last = {name: st.snapshot() for name, st in self.steppers.items()}
            epoch += 1
            reload_attempts = 0
            losses.next()

        return losses.val_best_losses, losses.best_loss_epoch
