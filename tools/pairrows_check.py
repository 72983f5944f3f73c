#!/usr/bin/env python
"""Monochrome conv pair in TF32 mode (the row-GEMM kernel, csrc/conv_pair_rows_tc.cu, where W % 4 == 0; the
TMEM-window kernel, csrc/conv_pair_tc.cu, otherwise): correctness against the FP32 CUDA-core kernel over ragged shapes,
then the time of the TF32 dispatch at batch 64.
    python tools/pairrows_check.py [--quick] [--multi] [--notime]
"""
import ctypes
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import univer_ocr_b200.nn as nn  # noqa: E402
from univer_ocr_b200._lib import ACT_LEAKY, ACT_NONE, ACT_SIGMOID, lib  # noqa: E402

nn.CP.use_gpu()
stream = nn.CP.stream()
rng = np.random.default_rng(5)


def event():
    e = ctypes.c_void_p()
    lib.uocr_event_create(ctypes.byref(e))
    return e.value


def run(d, y, n, h, w, mode, act1=ACT_LEAKY, act2=ACT_SIGMOID):
    lib.uocr_conv3x3_pair_fwd(d[0].ptr, d[1].ptr, d[2].ptr, d[3].ptr, d[4].ptr, y.ptr, n, h, w, 16,
                              act1, 0.01, act2, 0.0, mode, stream)


def problem(n, h, w):
    X = rng.uniform(size=(n, h, w, 1)).astype(np.float32)
    w1 = (rng.standard_normal((3, 3, 1, 16)) * 0.4).astype(np.float32)
    b1 = (rng.standard_normal(16) * 0.2).astype(np.float32)
    w2 = (rng.standard_normal((3, 3, 16, 1)) * 0.3).astype(np.float32)
    b2 = rng.standard_normal(1).astype(np.float32)
    return [nn.CP.copy(a) for a in (X, w1, b1, w2, b2)]


ok = True
shapes = [(2, 16, 32), (1, 5, 8), (3, 33, 244), (2, 40, 248), (2, 7, 492), (1, 64, 496), (3, 20, 736), (2, 496, 736),
          (1, 130, 1000), (5, 3, 12)]
if '--quick' in sys.argv:
    shapes = shapes[:4]
grids = [None, '1', '3'] if '--multi' in sys.argv else [None]
for g, (n, h, w) in [(g_, sh) for g_ in grids for sh in shapes]:
    if g is None:
        os.environ.pop('UOCR_PAIR_ROWS_GRID', None)
    else:
        os.environ['UOCR_PAIR_ROWS_GRID'] = g
    d = problem(n, h, w)
    for act1, act2 in ((ACT_LEAKY, ACT_SIGMOID), (ACT_LEAKY, ACT_NONE), (ACT_NONE, ACT_SIGMOID)):
        ref = nn.DeviceArray((n, h, w, 1))
        run(d, ref, n, h, w, 0, act1, act2)
        got = nn.DeviceArray.full((n, h, w, 1), -7.0)
        run(d, got, n, h, w, 1, act1, act2)
        a, b = got.get().astype(np.float64), ref.get().astype(np.float64)
        err = np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-30)
        bad = err > 2e-3
        ok &= not bad
        where = np.unravel_index(np.argmax(np.abs(a - b)), a.shape) if bad else ''
        print(f'{(n, h, w)} grid={g} act=({act1},{act2}): max err / max|ref| = {err:.2e} {"MISMATCH at " + str(where) if bad else "ok"}',
              flush=True)
print('ALL OK' if ok else 'FAILED', flush=True)

os.environ.pop('UOCR_PAIR_ROWS_GRID', None)
if '--notime' in sys.argv:
    sys.exit(0 if ok else 1)
n, h, w = 64, 496, 736
d = problem(n, h, w)
flush = nn.DeviceArray((64 * 1024 * 1024,))
y = nn.DeviceArray((n, h, w, 1))
for _ in range(3):
    run(d, y, n, h, w, 1)
ts = []
for _ in range(10):
    flush.fill(0)
    e0, e1 = event(), event()
    lib.uocr_event_record(e0, stream)
    run(d, y, n, h, w, 1)
    lib.uocr_event_record(e1, stream)
    lib.uocr_event_sync(e1)
    ms = ctypes.c_float(0)
    lib.uocr_event_elapsed_ms(e0, e1, ctypes.byref(ms))
    ts.append(ms.value)
t = float(np.median(ts))
print(f'tf32 pair: {t * 1e3:.1f} us per 64 tiles  ({186.9e6 / t / 1e6:.0f} GB/s algorithmic, '
      f'{186.9e6 / t / 1e6 / 6547.8 * 100:.1f} % of HBM peak)', flush=True)
