#!/usr/bin/env python
"""Ragged training steps against per-sample loops (Model.compute_loss_and_gradients_ragged).

    python tools/raggedtrainbench.py [--math tf32] [--lines 64] [--paragraphs 32]

For Char over L line crops of 32 x 40-900 and Line over P paragraph crops of 64-400 x 96-688 (multiples of 16, seeded
sizes), forward + loss + backward of the same samples
  loop:    one compute_loss_and_gradients per sample at batch 1 (the reference trains batch = 1);
  ragged:  one compute_loss_and_gradients_ragged over all of them on a zero-filled canvas;
and, on a batch of equal sizes (no padding), stacked compute_loss_and_gradients against
compute_loss_and_gradients_ragged with every extent equal to the canvas: the cost of the ragged bookkeeping.
Every input and target is on the device before timing.  Times are host clocks around work that ends in a stream
synchronise, after one warm-up call; two timed runs each.  Launches from uocr_launch_count.  Prints the card's name and
power limit with the numbers, and one JSON line per measurement.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

from textbench import card  # noqa: E402


def timed(fn, nn):
    from univer_ocr_b200._lib import launch_count
    nn.CP.synchronize()
    l0, t0 = launch_count(), time.perf_counter()
    fn()
    nn.CP.synchronize()
    return (time.perf_counter() - t0) * 1e3, launch_count() - l0


def targets_for(model, name, shape, rng):
    out = model.get_output_shapes([shape])[0]
    if name == 'char':
        y = np.zeros(out, np.float32)
        y[np.arange(out[0]), rng.integers(0, out[1], out[0])] = 1
        return y
    return (rng.uniform(size=out) < 0.3).astype(np.float32)


def case(name, sizes, nn, seed):
    """-> (model, per-sample device (X, y), device canvas, extents, device target canvas)."""
    from univer_ocr_b200 import my_model
    rng = np.random.default_rng(seed)
    model = my_model.MAKERS[name]((1, 32, 64, 1))
    ext = np.array(sizes, np.int64)
    H, W = ext.max(axis=0)
    canvas = np.zeros((len(ext), H, W, 1), np.float32)
    out_shape = model.get_output_shapes([canvas.shape])[0]
    y = np.zeros(out_shape, np.float32)
    samples = []
    for i, (h, w) in enumerate(ext):
        X = rng.uniform(0, 1, (1, h, w, 1)).astype(np.float32)
        t = targets_for(model, name, X.shape, rng)
        canvas[i, :h, :w] = X[0]
        if name == 'char':
            y[i * W:i * W + t.shape[0]] = t
        else:
            y[i, :t.shape[1], :t.shape[2]] = t[0]
        samples.append((nn.CP.copy(X), nn.CP.copy(t)))
    return model, samples, nn.CP.copy(canvas), ext, nn.CP.copy(y)


def measure(label, name, model, samples, canvas, ext, y, nn, stacked=False):
    if stacked:
        def loop():
            model.compute_loss_and_gradients(canvas, y)
    else:
        def loop():
            for X, t in samples:
                model.compute_loss_and_gradients(X, t)

    def ragged():
        model.compute_loss_and_gradients_ragged(canvas, ext, y)

    rows = []
    for kind, fn in ((('stacked' if stacked else 'loop'), loop), ('ragged', ragged)):
        fn()                                                    # warm-up: modules, plans, pools
        runs = [timed(fn, nn) for _ in range(2)]
        rows.append({'case': label, 'network': name, 'path': kind, 'images': len(ext),
                     'ms': [round(r[0], 2) for r in runs], 'launches': runs[0][1]})
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--math', default='tf32', choices=['fp32', 'tf32'])
    ap.add_argument('--lines', type=int, default=64)
    ap.add_argument('--paragraphs', type=int, default=32)
    args = ap.parse_args()
    import univer_ocr_b200.nn as nn
    nn.CP.use_gpu()
    nn.CP.set_math_mode(args.math)
    print(f'card: {card()}  math: {args.math}')
    rng = np.random.default_rng(7)
    char_sizes = [(32, int(w)) for w in rng.integers(40, 901, args.lines)]
    line_sizes = [(int(rng.integers(4, 26)) * 16, int(rng.integers(6, 44)) * 16) for _ in range(args.paragraphs)]
    rows = []
    for name, sizes, even in (('char', char_sizes, [(32, 400)] * args.lines),
                              ('line', line_sizes, [(256, 384)] * args.paragraphs)):
        rows += measure('mixed sizes', name, *case(name, sizes, nn, 1), nn)
        rows += measure('no padding', name, *case(name, even, nn, 2), nn, stacked=True)
    for r in rows:
        print(f"{r['network']:5s} {r['case']:12s} {r['path']:8s} {r['images']:3d} images: "
              f"{' / '.join(f'{m:.2f}' for m in r['ms'])} ms, {r['launches']} launches")
    for r in rows:
        print(json.dumps({**r, 'math': args.math, 'card': card()}))


if __name__ == '__main__':
    main()
