#!/usr/bin/env python
"""Ragged batches against per-item loops (Model.predict_ragged, TextPipeline.batch).

    python tools/textbench.py [--repeat 3] [--math tf32]

(a) The networks alone: Line over P = 128 paragraph crops of 64-400 x 96-700 and Char over L = 1024 lines of width
    40-900 (seeded sizes), as a loop of Model.predict calls and as one ragged call.
(b) The whole pipeline: TextPipeline.batch against a loop of TextPipeline.__call__ on 64 pages of 496 x 736.  The
    Monochrome / Paragraph / Line maps are deterministic stand-ins built like tests/stage_cases.py, so the paragraph and
    line counts are fixed; Char is the real network.
Times are host clocks around work that ends in a stream synchronise; launches from uocr_launch_count; read-backs are
device-to-host copies.  Prints the card's name and power limit with the numbers, and one JSON line per run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else 'unknown'
    except (OSError, subprocess.SubprocessError):
        return 'unknown'


class Counter:
    """Counts launches, model builds and device-to-host copies over a `with` block."""

    def __init__(self):
        from univer_ocr_b200 import my_model
        from univer_ocr_b200._lib import lib
        self.lib, self.makers = lib, my_model.MAKERS

    def __enter__(self):
        from univer_ocr_b200._lib import launch_count
        self.builds = self.reads = 0
        self.saved_makers = dict(self.makers)
        for name, make in self.saved_makers.items():
            def counted(*a, _make=make, **k):
                self.builds += 1
                return _make(*a, **k)
            self.makers[name] = counted
        self.lib.load()
        d2h = self.saved_d2h = self.lib.uocr_memcpy_d2h

        def counted_d2h(*a):
            self.reads += 1
            return d2h(*a)
        self.lib.uocr_memcpy_d2h = counted_d2h
        self.launches0 = launch_count()
        self.t0 = time.perf_counter()
        return self

    def __exit__(self, *exc):
        from univer_ocr_b200._lib import launch_count
        import univer_ocr_b200.nn as nn
        nn.CP.synchronize()
        self.seconds = time.perf_counter() - self.t0
        self.launches = launch_count() - self.launches0
        self.makers.update(self.saved_makers)
        self.lib.uocr_memcpy_d2h = self.saved_d2h


def part_a(args, nn):
    from univer_ocr_b200 import predict
    rng = np.random.default_rng(7)
    crops = [rng.uniform(0, 1, (1, int(rng.integers(4, 26)) * 16, int(rng.integers(6, 44)) * 16, 1)).astype(np.float32)
             for _ in range(args.paragraphs)]
    lines = [rng.uniform(0, 1, (1, 32, int(rng.integers(40, 901)), 1)).astype(np.float32) for _ in range(args.lines)]
    crops, lines = [nn.CP.copy(c) for c in crops], [nn.CP.copy(x) for x in lines]
    rows = []
    for rep in range(args.repeat + 1):                       # the first pass builds the models and warms every shape
        for name, items in (('line', crops), ('char', lines)):
            pipe = predict.TextPipeline()
            pipe.predict(name, items[0])
            with Counter() as loop:
                for x in items:
                    pipe.predict(name, x)
            mult = pipe.CHAR_WIDTH_MULTIPLE if name == 'char' else 1
            pipe._ragged(name, items, mult)
            with Counter() as one:
                pipe._ragged(name, items, mult)
            if rep:
                rows.append({'part': 'a', 'network': name, 'items': len(items),
                             'loop_ms': round(loop.seconds * 1e3, 3), 'ragged_ms': round(one.seconds * 1e3, 3),
                             'loop_launches': loop.launches, 'ragged_launches': one.launches,
                             'loop_builds': loop.builds, 'ragged_builds': one.builds})
    return rows


def part_b(args, nn):
    from oracle import np_oracle as O
    from tests import stage_cases as C
    from univer_ocr_b200 import predict
    pages, preds = [], {}
    for k in range(args.pages):
        pred, images = C.paragraph_page(k % 4, h=496, w=736, tilt=((12.0, -25.0), (80.0, 3.0), (5.0, 40.0),
                                                                    (-30.0, 10.0))[k % 4])
        pages.append(images[0])
        preds[k % 4] = nn.CP.copy(O.make_divisible_by(pred, 16, 16).astype(np.float32))

    state = {'page': 0}

    def paragraph(x):                                         # the stand-in map of the page being read
        out = preds[state['page'] % 4]
        state['page'] += 1
        return out

    def lines_for(x):
        _, h, w, _ = x.shape
        out = np.zeros((1, h, w, 2), np.float32)
        for centre in range(h // 6, h - 10, 24):
            out[0, max(centre - 6, 0):centre - 4, 6:w - 6, 0] = 1.0
            out[0, centre + 4:centre + 6, 6:w - 6, 1] = 1.0
        return nn.CP.copy(out)

    stand = {'monochrome': lambda x: x, 'paragraph': paragraph, 'line': lines_for}
    pipe = predict.TextPipeline(predictors=stand)
    dev_pages = [nn.CP.copy(p) for p in pages]
    rows = []
    for rep in range(args.repeat + 1):
        state['page'] = 0
        with Counter() as loop:
            want = [pipe(p) for p in dev_pages]
        state['page'] = 0
        with Counter() as one:
            got = pipe.batch(dev_pages)
        n_lines = sum(len(p) for r in got for p in r['text'])
        assert n_lines == sum(len(p) for r in want for p in r['text'])
        if rep:
            rows.append({'part': 'b', 'pages': len(pages), 'lines': n_lines,
                         'loop_pages_per_s': round(len(pages) / loop.seconds, 2),
                         'batch_pages_per_s': round(len(pages) / one.seconds, 2),
                         'loop_launches_per_page': round(loop.launches / len(pages), 1),
                         'batch_launches_per_page': round(one.launches / len(pages), 1),
                         'loop_reads_per_page': round(loop.reads / len(pages), 2),
                         'batch_reads_per_page': round(one.reads / len(pages), 2)})
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--repeat', type=int, default=3)
    ap.add_argument('--math', default='tf32')
    ap.add_argument('--paragraphs', type=int, default=128)
    ap.add_argument('--lines', type=int, default=1024)
    ap.add_argument('--pages', type=int, default=64)
    args = ap.parse_args()
    import univer_ocr_b200.nn as nn
    nn.CP.use_gpu()
    nn.CP.set_math_mode(args.math)
    gpu = card()
    for row in part_a(args, nn) + part_b(args, nn):
        print(json.dumps({'gpu': gpu, 'math': args.math, **row}), flush=True)


if __name__ == '__main__':
    main()
