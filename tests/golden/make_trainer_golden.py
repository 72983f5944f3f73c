"""Generates tests/golden/trainer_traces.json by running the UNMODIFIED reference epoch driver
(`my_model/trainer.py`) over the scripted scenarios of tests/trainer_cases.py.  Needs a
checkout of the reference:

    UOCR_REFERENCE_ROOT=<reference checkout> python tests/golden/make_trainer_golden.py
"""
import contextlib
import io
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import ref_loader  # noqa: E402
from tests import trainer_cases  # noqa: E402


def main():
    ref = ref_loader.load_trainer()
    out = {}
    for name in trainer_cases.SCENARIOS:
        with contextlib.redirect_stdout(io.StringIO()):
            out[name] = trainer_cases.run(name, trainer_cases.reference_factory(ref))
        print(name, len(out[name]['trace']), 'events, best', out[name]['best'], out[name]['best_epoch'])
    with open(os.path.join(HERE, 'trainer_traces.json'), 'w') as fp:
        json.dump(out, fp, indent=0, separators=(',', ':'))


if __name__ == '__main__':
    main()
