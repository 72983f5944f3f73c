#!/usr/bin/env python
"""Monochrome conv pair: TF32 tensor-core kernel vs the FP32 CUDA-core kernel (correctness + time).
    python tools/pairbench.py [--batch 64] [--iters 10] [--h 496] [--w 736]
"""
import argparse
import ctypes
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=64)
    ap.add_argument('--iters', type=int, default=10)
    ap.add_argument('--h', type=int, default=496)
    ap.add_argument('--w', type=int, default=736)
    args = ap.parse_args()
    import univer_ocr_b200.nn as nn
    from univer_ocr_b200._lib import ACT_LEAKY, ACT_SIGMOID, lib
    nn.CP.use_gpu()
    stream = nn.CP.stream()
    rng = np.random.default_rng(5)
    n, h, w = args.batch, args.h, args.w
    X = rng.uniform(size=(n, h, w, 1)).astype(np.float32)
    w1 = (rng.standard_normal((3, 3, 1, 16)) * 0.4).astype(np.float32)
    b1 = (rng.standard_normal(16) * 0.2).astype(np.float32)
    w2 = (rng.standard_normal((3, 3, 16, 1)) * 0.3).astype(np.float32)
    b2 = rng.standard_normal(1).astype(np.float32)
    d = [nn.CP.copy(a) for a in (X, w1, b1, w2, b2)]
    flush = nn.DeviceArray((64 * 1024 * 1024,))

    def event():
        e = ctypes.c_void_p()
        lib.uocr_event_create(ctypes.byref(e))
        return e.value

    outs = {}
    for mode in (0, 1):
        y = nn.DeviceArray((n, h, w, 1))

        def run():
            rc = lib.uocr_conv3x3_pair_fwd(d[0].ptr, d[1].ptr, d[2].ptr, d[3].ptr, d[4].ptr, y.ptr, n, h, w, 16,
                                           ACT_LEAKY, 0.01, ACT_SIGMOID, 0.0, mode, stream)
            assert rc == 0, rc
        run()
        run()
        ts = []
        for _ in range(args.iters):
            flush.fill(0)
            e0, e1 = event(), event()
            lib.uocr_event_record(e0, stream)
            run()
            lib.uocr_event_record(e1, stream)
            lib.uocr_event_sync(e1)
            ms = ctypes.c_float(0)
            lib.uocr_event_elapsed_ms(e0, e1, ctypes.byref(ms))
            ts.append(ms.value)
        outs[mode] = np.asarray(y.get(), dtype=np.float64)
        px = n * h * w
        med = float(np.median(ts))
        print(f'mode {"tf32" if mode else "fp32"}: median {med:.4f} ms  best {min(ts):.4f} ms  '
              f'{8 * px / med / 1e6:.0f} GB/s  {2 * 288 * px / med / 1e9:.1f} TFLOP/s', flush=True)
    err = np.abs(outs[1] - outs[0])
    print(f'max |tf32 - fp32| = {err.max():.3e} (mean {err.mean():.3e}, signed mean {(outs[1] - outs[0]).mean():.3e})')
    bad = np.argwhere(err > 2e-3)
    if len(bad):
        print('mismatches:', len(bad), 'first', bad[:10].tolist())
        sys.exit(1)


if __name__ == '__main__':
    main()
