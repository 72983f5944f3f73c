"""TEST INFRASTRUCTURE ONLY -- loader for the *unmodified* reference (KerkDovan/univer-ocr).

Imports the reference's `web_app.components.nn` (and `my_model.model`) straight from the
checkout that `UOCR_REFERENCE_ROOT` names, under a handful of compatibility shims, so that its
NumPy CPU path can be executed to (a) pin `oracle/np_oracle.py` and (b) generate the golden
vectors committed under `tests/golden/`.

The reference is not part of this repository: without `UOCR_REFERENCE_ROOT` pointing at a
checkout of it, `available()` returns False and the live comparisons skip (the committed
golden vectors keep checking what they recorded).

Why shims are needed (reference targets Python 3.7 / NumPy 1.18 / CuPy 7):
  * `import cupy` at module top            -- nn/gpu.py:1, nn/gradient_check.py:3
  * `from collections import Iterable`     -- nn/help_func.py:1
  * `np.product`, `np.float`, `np.bool`    -- nn/layers/layers.py:298, nn/regularizations.py:6,
                                              nn/layers/maxpool.py:144
  * `web_app/__init__.py` imports Flask; `image_generator/generate.py:7` imports Faker
Nothing in the reference tree is modified or copied.
"""
import collections
import collections.abc
import importlib
import os
import sys
import types

import numpy as np

REFERENCE_ROOT = os.environ.get('UOCR_REFERENCE_ROOT', '')

_loaded = {}


def available():
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, 'web_app', 'components', 'nn'))


def _install_shims():
    if not hasattr(collections, 'Iterable'):
        collections.Iterable = collections.abc.Iterable
    for name, repl in (('product', np.prod), ('float', float), ('bool', bool)):
        if name not in np.__dict__:
            setattr(np, name, repl)
    if 'cupy' not in sys.modules:
        try:
            importlib.import_module('cupy')
        except Exception:
            stub = types.ModuleType('cupy')
            stub.asarray = np.asarray
            stub.asnumpy = np.asarray
            stub.ndarray = np.ndarray
            stub.__uocr_stub__ = True
            sys.modules['cupy'] = stub
    if 'faker' not in sys.modules:
        try:
            importlib.import_module('faker')
        except Exception:
            stub = types.ModuleType('faker')
            stub.Faker = object
            sys.modules['faker'] = stub
    # Empty package shells so that `web_app/__init__.py` (Flask app) is never executed.
    for pkg, rel in (('web_app', 'web_app'), ('web_app.components', 'web_app/components')):
        if pkg not in sys.modules:
            mod = types.ModuleType(pkg)
            mod.__path__ = [os.path.join(REFERENCE_ROOT, rel)]
            sys.modules[pkg] = mod


def load_nn():
    """Returns the reference's `web_app.components.nn` package (NumPy CPU mode)."""
    if 'nn' in _loaded:
        return _loaded['nn']
    if not available():
        raise RuntimeError(f'reference tree not found at {REFERENCE_ROOT!r}: set UOCR_REFERENCE_ROOT to a checkout of it')
    _install_shims()
    nn = importlib.import_module('web_app.components.nn')
    for sub in ('gpu', 'layers', 'losses', 'optimizers', 'regularizations', 'initializers',
                'models', 'gradient_check'):
        importlib.import_module(f'web_app.components.nn.{sub}')
    nn.gpu.CP.use_cpu()
    _loaded['nn'] = nn
    return nn


def load_my_model():
    """Returns the reference's `web_app.components.my_model.model` module."""
    if 'my_model' in _loaded:
        return _loaded['my_model']
    load_nn()
    mod = importlib.import_module('web_app.components.my_model.model')
    _loaded['my_model'] = mod
    return mod


def load_trainer():
    """Returns the reference's `web_app.components.my_model.trainer` module (epoch driver:
    `Losses`, `Trainer`).  Pure Python + NumPy + tqdm, no shims beyond the package shells."""
    if 'trainer' in _loaded:
        return _loaded['trainer']
    if not available():
        raise RuntimeError(f'reference tree not found at {REFERENCE_ROOT!r}: set UOCR_REFERENCE_ROOT to a checkout of it')
    _install_shims()
    mod = importlib.import_module('web_app.components.my_model.trainer')
    _loaded['trainer'] = mod
    return mod


def load_my_model_on(nn_package, alias='uocr_dropin'):
    """The reference's UNMODIFIED `my_model/model.py` (and `nn/model_system.py`, `interpreter/`) imported a second
    time, under the package name `<alias>.components`, with `..nn` resolving to `nn_package` (e.g.
    `univer_ocr_b200.nn`) wherever that package has a module of the same name, and to the reference's own file
    otherwise (model_system.py, which only orchestrates).  This is route A of INTEGRATION.md executed literally:
    the reference's builders construct their networks out of the drop-in layer classes.

    Returns the imported `<alias>.components.my_model.model` module."""
    key = f'dropin:{alias}'
    if key in _loaded:
        return _loaded[key]
    if not available():
        raise RuntimeError(f'reference tree not found at {REFERENCE_ROOT!r}: set UOCR_REFERENCE_ROOT to a checkout of it')
    _install_shims()
    comp_dir = os.path.join(REFERENCE_ROOT, 'web_app', 'components')
    for pkg, path in ((alias, os.path.join(REFERENCE_ROOT, 'web_app')), (f'{alias}.components', comp_dir)):
        mod = types.ModuleType(pkg)
        mod.__path__ = [path]
        sys.modules[pkg] = mod
    nn_alias = types.ModuleType(f'{alias}.components.nn')
    nn_alias.__path__ = [os.path.join(comp_dir, 'nn')]             # fallback: the reference's own files
    sys.modules[nn_alias.__name__] = nn_alias
    prefix = nn_package.__name__ + '.'
    for name, module in list(sys.modules.items()):
        if name.startswith(prefix) and module is not None:
            sub = name[len(prefix):]
            sys.modules[f'{nn_alias.__name__}.{sub}'] = module      # the drop-in's module wins
            if '.' not in sub:
                setattr(nn_alias, sub, module)
    mod = importlib.import_module(f'{alias}.components.my_model.model')
    _loaded[key] = mod
    return mod
