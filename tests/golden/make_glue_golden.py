"""Generates tests/golden/glue.json by running the UNMODIFIED reference's PredToText._func1
(interpreter/interpreter.py:595-614) and make_divisible_by (my_model/model.py:26-34) on seeded
inputs.  The alphabet and the similar-character table are read from the reference's
`primitives` package at generation time and stored as fixture data.  Needs a checkout of the reference:

    UOCR_REFERENCE_ROOT=<reference checkout> python tests/golden/make_glue_golden.py
"""
import importlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import ref_loader  # noqa: E402


def main():
    ref_loader.load_nn()
    interp = importlib.import_module('web_app.components.interpreter.interpreter')
    prim = importlib.import_module('web_app.components.primitives')
    model = ref_loader.load_my_model()
    chars = prim.CHARS
    similar = {k: sorted(v) for k, v in prim.SIMILAR_CHARS.items()}
    rng = np.random.default_rng(99)
    cases = []
    for rows, style in ((40, 'softmax'), (64, 'ties'), (25, 'zeros')):
        pred = rng.standard_normal((rows, len(chars))).astype(np.float32)
        if style == 'softmax':
            e = np.exp(pred * 3)
            pred = (e / e.sum(axis=1, keepdims=True)).astype(np.float32)
        elif style == 'ties':
            pred = (np.round(pred * 2) / 2).astype(np.float32)      # many exact ties
            pred[::5, 0] = 9.0                                       # blanks reset the repeat filter
        else:
            pred = np.abs(pred)
            pred[::3, :] = 0.0                                       # all-zero rows emit nothing
            pred[1::3, 17] = 50.0
            pred[2::3, 17] = 50.0                                    # repeated winner collapses
        text = interp.PredToText._func1(pred.astype(np.float64))
        cases.append({'pred': pred.tolist(), 'text': text})
    pads = []
    for shape in ((1, 480, 720, 1), (2, 33, 47, 3), (1, 16, 32, 1)):
        out = model.make_divisible_by(np.ones(shape), 16, 16)
        ys, xs = np.nonzero(out[0, :, :, 0])
        pads.append({'shape': list(shape), 'out_shape': list(out.shape),
                     'top': int(ys.min()), 'left': int(xs.min())})
    with open(os.path.join(HERE, 'glue.json'), 'w') as fp:
        json.dump({'chars': chars, 'similar': similar, 'pred_to_text': cases, 'make_divisible_by': pads}, fp)
    print([c['text'] for c in cases], pads)


if __name__ == '__main__':
    main()
