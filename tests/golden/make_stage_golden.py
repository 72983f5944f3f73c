"""Generates tests/golden/stages.npz by running the UNMODIFIED reference's crop-stage functions
(interpreter/interpreter.py: label_layer :16-22, rearrange_lines :41-84, rotate_array :188-192,
FindObjectHeightInRotated._func :229-232, CropRotateAndZoomLines._func1 / _func2 :493-523, the ternary search of
CropAndRotateSingleParagraph._func :318-343) on the seeded synthetic cases of tests/stage_cases.py.  Inputs are not
stored: tests regenerate them from the same seeds.  Needs a checkout of the reference:

    UOCR_REFERENCE_ROOT=<reference checkout> python tests/golden/make_stage_golden.py

Boolean masks are cast to uint8 before the reference's own `ndimage.find_objects` calls (SciPy >= 1.18 refuses a boolean
maximum label; the boxes are the same).  Arrays are handed over as float32, so the reference's float32 results are the
bits the device must reproduce."""
import importlib
import os
import sys

import numpy as np
from scipy import ndimage

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import ref_loader  # noqa: E402
from tests import stage_cases as C  # noqa: E402

ZOOMED, MINIMAL = 32, 200


def main():
    ref_loader.load_my_model()
    I = importlib.import_module('web_app.components.interpreter.interpreter')
    out = {}

    def u8(m):
        return m.astype(np.uint8)

    def thresholded(arr):                                    # interpreter.py:437-438 (a closure there)
        return arr > 0.5 * (np.mean(arr) + np.max(arr))

    for direction in (None, 90, 180, 270):
        mask, arrays = C.line_paragraph(1, direction)
        top, bottom = thresholded(mask[..., 0:1]), thresholded(mask[..., 1:2])
        tops, bottoms, rotation = I.rearrange_lines(I.label_layer(top), I.label_layer(bottom))
        assert rotation == direction
        tag = f'lines_{direction}'
        out[f'{tag}__count'] = np.int64(len(tops))
        for lid, (t, b) in enumerate(zip(tops, bottoms)):
            y, x = I.CropRotateAndZoomLines._func1(u8(t), u8(b))
            out[f'{tag}__box{lid}'] = np.array([y.start, y.stop, x.start, x.stop], np.int64)
            for aid, arr in enumerate(arrays):
                out[f'{tag}__line{lid}_array{aid}'] = I.CropRotateAndZoomLines._func2(arr, y, x, rotation, ZOOMED, MINIMAL)
    for seed, tilt in ((0, (12.0, -25.0)), (1, (80.0, 3.0))):
        pred, images = C.paragraph_page(seed, tilt=tilt)
        objects = I.label_layer(pred)
        tag = f'page_{seed}'
        out[f'{tag}__count'] = np.int64(len(objects))
        for pid, m in enumerate(objects):
            _, ry, rx, _ = ndimage.find_objects(u8(m))[0]
            cm = u8(m[:, ry, rx, :])
            low, high = 0.0, 180.0
            while high - low > 1.0:                          # CropAndRotateSingleParagraph._func, :318-333
                a, b = low + (high - low) / 3, high - (high - low) / 3
                if I.FindObjectHeightInRotated._func(cm, a) < I.FindObjectHeightInRotated._func(cm, b):
                    high = b
                else:
                    low = a
            angle = (high + low) / 2
            assert 1.0 <= angle <= 179.0
            out[f'{tag}__angle{pid}'] = np.float64(angle)
            _, oy, ox, _ = ndimage.find_objects(I.rotate_array(cm, angle, good_rotation=False))[0]
            for iid, image in enumerate(images):
                out[f'{tag}__par{pid}_image{iid}'] = I.rotate_array((image * m)[:, ry, rx, :], angle)[:, oy, ox, :]
    path = os.path.join(HERE, 'stages.npz')
    np.savez_compressed(path, **out)
    print(path, len(out), 'arrays', os.path.getsize(path), 'bytes')


if __name__ == '__main__':
    main()
