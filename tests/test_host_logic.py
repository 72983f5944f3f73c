"""CPU-only checks: the C ABI exports every symbol include/uocr.h declares, the product refuses
to run without a GPU (no CPU fallback), and the host-side logic that needs no device (argument
helpers, shape arithmetic, graph flattening / ordering / fusion planning, receptive fields)
matches the reference's behaviour."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import np_oracle as O, ref_loader

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def built_lib():
    from univer_ocr_b200 import build
    path = build.build()
    assert os.path.exists(path)
    return path


def test_abi_exports_every_declared_symbol(built_lib):
    from univer_ocr_b200 import _lib
    protos = _lib.parse_header()
    assert len(protos) >= 60
    out = subprocess.run(['nm', '-D', '--defined-only', built_lib], capture_output=True, text=True).stdout
    exported = {line.split()[-1] for line in out.splitlines() if ' T ' in line}
    missing = sorted(set(protos) - exported)
    assert not missing, f'declared in uocr.h but not exported: {missing}'
    extra = sorted(n for n in exported if n.startswith('uocr_') and n not in protos)
    assert not extra, f'exported but undeclared: {extra}'
    dll = ctypes.CDLL(built_lib)
    for name in protos:
        assert getattr(dll, name) is not None
    assert _lib.lib.uocr_version() == 100                       # loads, no compute call


def test_conv_desc_struct_matches_header():
    from univer_ocr_b200._lib import ConvDesc
    text = open(os.path.join(ROOT, 'include', 'uocr.h')).read()
    body = text[text.index('typedef struct uocr_conv2d_desc'):text.index('} uocr_conv2d_desc;')]
    import re
    body = re.sub(r'/\*.*?\*/', '', body, flags=re.S)
    names = []
    for decl in re.findall(r'(?:int64_t|int32_t|float)\s+([^;]+);', body):
        names += [n.strip() for n in decl.split(',')]
    assert names == [f[0] for f in ConvDesc._fields_]
    assert ctypes.sizeof(ConvDesc) == 5 * 8 + 6 * 4 + 4 + 4 + 4 + 4


def test_no_cpu_fallback():
    import torch  # noqa: F401  (only to learn whether a GPU is visible here)
    from univer_ocr_b200 import _lib
    from univer_ocr_b200.nn import CP
    with pytest.raises(RuntimeError):
        CP.use_cpu()
    if _lib.device_count() == 0:
        with pytest.raises(_lib.UocrError):
            _lib.require_device()
        with pytest.raises(_lib.UocrError):
            CP.copy(np.zeros((2, 2)))
    # the product package never imports the oracle
    for dirpath, _, files in os.walk(os.path.join(ROOT, 'univer_ocr_b200')):
        for f in files:
            if f.endswith('.py'):
                src = open(os.path.join(dirpath, f)).read()
                assert 'import oracle' not in src and 'from oracle' not in src, f


def test_tuplize_semantics():
    from univer_ocr_b200.nn.help_func import make_list_if_not, tuplize
    assert tuplize('k', 3, 2) == (3, 3) and tuplize('k', (2, 5), 2) == (2, 5) and tuplize('k', [1, 2], 2) == (1, 2)
    with pytest.raises(ValueError):
        tuplize('k', -1, 2)
    with pytest.raises(ValueError):
        tuplize('k', (1, -2), 2)
    for bad in ((1, 2, 3), 'ab', 1.5, (1.0, 2)):
        with pytest.raises(TypeError):
            tuplize('k', bad, 2)
    assert make_list_if_not(1) == [1] and make_list_if_not([1]) == [1] and make_list_if_not((1,)) == [(1,)]


def _layers():
    from univer_ocr_b200.nn import layers
    return layers


def test_output_shape_arithmetic_matches_oracle():
    L = _layers()
    rng = np.random.default_rng(0)
    for _ in range(200):
        h, w = int(rng.integers(1, 40)), int(rng.integers(1, 40))
        k = (int(rng.integers(1, 6)), int(rng.integers(1, 6)))
        p = (int(rng.integers(0, 3)), int(rng.integers(0, 3)))
        s = (int(rng.integers(1, 4)), int(rng.integers(1, 4)))
        if h + 2 * p[0] < k[0] or w + 2 * p[1] < k[1]:
            continue
        conv = L.Convolutional2D(k, out_channels=5, padding=p, stride=s)     # un-initialised: no device
        assert conv.get_output_shapes((2, h, w, 3))[0] == (2, *O.conv2d_out_hw(h, w, k, p, s), 5)
        for ceil in (False, True):
            pool = L.MaxPool2D(k, padding=p, stride=s, ceil_mode=ceil)
            assert pool.get_output_shapes((2, h, w, 3))[0] == (2, *O.maxpool2d_out_hw(h, w, k, p, s, ceil), 3)
    assert L.Upsample2D((2, 3)).get_output_shapes((4, 5, 6, 7)) == [(4, 10, 18, 7)]
    assert L.Conv2DToBatchedFixedWidthed(8).get_output_shapes((3, 1, 20, 64)) == [(60, 1, 8, 64)]
    with pytest.raises(AssertionError):
        L.Conv2DToBatchedFixedWidthed(8).get_output_shapes((3, 1, 7, 64))
    assert L.Flatten().get_output_shapes((6, 1, 8, 64)) == [(6, 512)]
    assert L.Concat().get_output_shapes([(2, 4, 4, 3), (2, 4, 4, 5)]) == [(2, 4, 4, 8)]


def _uninitialised_paragraph():
    """make_paragraph's topology (my_model/model.py:137-191) from un-initialised layers, so no
    device is touched."""
    L = _layers()
    from univer_ocr_b200.nn.models import Model

    def block(stride, sigmoid=False):
        return Model({'conv_1': L.Convolutional2D((5, 5), out_channels=1, padding=2, stride=stride),
                      ('sigmoid' if sigmoid else 'leaky_relu_1'): (L.Sigmoid() if sigmoid else L.LeakyRelu(0.01))},
                     {'conv_1': 0, ('sigmoid' if sigmoid else 'leaky_relu_1'): 'conv_1',
                      0: ('sigmoid' if sigmoid else 'leaky_relu_1')})

    def up():
        return Model({'upsample': L.Upsample2D(2), 'conv_block': block(1)},
                     {'upsample': 0, 'conv_block': 'upsample', 0: 'conv_block'})
    inner = Model({'down_1': block(2), 'down_2': block(2), 'up_1': up(), 'up_2': up(), 'end': block(1, True)},
                  {'down_1': 0, 'down_2': 'down_1', 'up_2': 'down_2', 'up_1': 'up_2', 'end': 'up_1', 0: 'end'})
    return Model({'Paragraph': inner}, {'Paragraph': 0, 0: 'Paragraph'})


def test_nested_model_flattening_order_and_fusion_plan():
    model = _uninitialised_paragraph()
    assert list(model.layers) == [
        'Paragraph/down_1/conv_1', 'Paragraph/down_1/leaky_relu_1', 'Paragraph/down_2/conv_1',
        'Paragraph/down_2/leaky_relu_1', 'Paragraph/up_1/upsample', 'Paragraph/up_1/conv_block/conv_1',
        'Paragraph/up_1/conv_block/leaky_relu_1', 'Paragraph/up_2/upsample',
        'Paragraph/up_2/conv_block/conv_1', 'Paragraph/up_2/conv_block/leaky_relu_1',
        'Paragraph/end/conv_1', 'Paragraph/end/sigmoid']
    assert model.relations['Paragraph/down_1/conv_1'] == [0]
    assert model.relations['Paragraph/up_2/upsample'] == ['Paragraph/down_2/leaky_relu_1']
    assert model.relations['Paragraph/end/conv_1'] == ['Paragraph/up_1/conv_block/leaky_relu_1']
    assert model.relations[0] == ['Paragraph/end/sigmoid']
    order = model._resolve_order()
    assert order[0] == 'Paragraph/down_1/conv_1' and order[-1] == 'Paragraph/end/sigmoid'
    assert order.index('Paragraph/up_2/upsample') < order.index('Paragraph/up_1/upsample')
    # plans need relations_backward; build it the way initialize() does, without touching layers
    model._order = order
    for name in order + [0]:
        for i, src in enumerate(model.relations[name]):
            model.relations_backward.setdefault(src, {})[name] = i
    for layer in model.layers.values():
        if hasattr(layer, 'in_channels'):
            layer.in_channels = 1
    infer = model._make_plan(training=False)
    train = model._make_plan(training=True)
    assert [s[0] for s in infer] == ['conv'] * 5
    assert infer[2] == ('conv', 'Paragraph/up_2/upsample', 'Paragraph/up_2/conv_block/conv_1',
                        'Paragraph/up_2/conv_block/leaky_relu_1')
    assert infer[4] == ('conv', None, 'Paragraph/end/conv_1', 'Paragraph/end/sigmoid')
    # training: conv+LeakyRelu fuse; the upsample folds into the 5x5 1->1 conv (its wgrad kernel reads
    # through the upsampling); the final Sigmoid stays a separate layer
    assert ('conv', 'Paragraph/up_1/upsample', 'Paragraph/up_1/conv_block/conv_1',
            'Paragraph/up_1/conv_block/leaky_relu_1') in train
    assert ('layer', 'Paragraph/end/sigmoid') in train
    assert ('conv', None, 'Paragraph/end/conv_1', None) not in train
    assert ('conv', None, 'Paragraph/down_1/conv_1', 'Paragraph/down_1/leaky_relu_1') in train


def test_receptive_field_matches_reference_values():
    """SURVEY.md 5: receptive field 29x29 for the Paragraph / Line topology."""
    model = _uninitialised_paragraph()
    model._order = model._resolve_order()
    model.is_initialized = True
    rf = model.get_receptive_fields()
    end = rf['Paragraph/end/conv_1']['input 0']
    assert end['cnt'] == (29, 29) and end['is_solid_y'] and end['is_solid_x']
    assert rf['Paragraph/down_1/conv_1']['input 0']['cnt'] == (5, 5)


@pytest.mark.skipif(not ref_loader.available(), reason='needs the reference tree (UOCR_REFERENCE_ROOT)')
def test_flattening_matches_reference_model():
    """Same nested construction through the reference's own Model: identical leaf names,
    relations and receptive fields."""
    mm = ref_loader.load_my_model()
    ref = mm.make_paragraph((1, 32, 32, 1))
    mine = _uninitialised_paragraph()
    assert list(ref.layers) == list(mine.layers)
    assert {k: list(v) for k, v in ref.relations.items()} == mine.relations
    mine._order = mine._resolve_order()
    mine.is_initialized = True
    assert ref.get_receptive_fields() == mine.get_receptive_fields()


@pytest.mark.parametrize('name', ['monochrome', 'paragraph', 'line', 'char'])
def test_builders_match_reference_parameters_golden(golden, name):
    """What the reference's own builders produced, as tests/golden/models.npz recorded it (make_golden.py builds each
    network with the reference's make_*): every parameter's flattened name, in the reference's order, and the
    network's output shape.  my_model's builders must give the same, with no device."""
    import univer_ocr_b200.nn as nn
    from tests.cases import MODEL_SHAPES
    from univer_ocr_b200 import my_model
    g = golden('models').case(name)
    want = [k[len('grad1__'):-len('__val')] for k in g if k.startswith('grad1__') and k.endswith('__val')]
    shape = MODEL_SHAPES[name]
    model = my_model.MAKERS[name](shape, optimizer=nn.optimizers.Adam(lr=0.0015))
    assert [k.replace('/', '.') for k in model.params()] == want and len(want) >= 4
    assert tuple(model.get_output_shapes([shape])[0]) == g['pred0'].shape


def test_multi_output_submodel_tuple_sources():
    """(name, i, j) sources select outputs of a nested multi-output model (models.py:136-139)."""
    L = _layers()
    from univer_ocr_b200.nn.models import Model
    two = Model({'a': L.Noop(), 'b': L.Relu()}, {'a': 0, 'b': 0, 0: 'a', 1: 'b'})
    outer = Model({'two': two, 'cat': L.Concat(), 'only_b': L.Noop()},
                  {'two': 0, 'cat': 'two', 'only_b': ('two', 1), 0: 'cat', 1: 'only_b'})
    assert outer.relations['cat'] == ['two/a', 'two/b']
    assert outer.relations['only_b'] == ['two/b']
    assert outer.relations['two/a'] == [0] and outer.relations['two/b'] == [0]
    assert outer.inputs_count == 1 and outer.outputs_count == 2
    with pytest.raises(TypeError):
        Model([L.Noop()], {})
    from univer_ocr_b200.nn.models import Sequential
    seq = Sequential([L.Noop(), L.Relu()])
    assert list(seq.layers) == ['0_Noop', '1_Relu'] and seq.relations[0] == ['1_Relu']


def test_make_divisible_by_and_weights_json_format(tmp_path):
    from univer_ocr_b200.my_model import make_divisible_by
    a = np.arange(2 * 16 * 30, dtype=np.float64).reshape(2, 16, 30, 1)
    assert np.array_equal(make_divisible_by(a, 16, 16), O.make_divisible_by(a, 16, 16))
    b = np.ones((1, 17, 33, 1))
    assert make_divisible_by(b, 16, 16).shape == (1, 32, 48, 1)
    assert np.array_equal(make_divisible_by(b, 16, 16), O.make_divisible_by(b, 16, 16))


def test_progress_tracker_protocol():
    from univer_ocr_b200.nn.progress_tracker import ProgressTracker, track_method
    events = []
    tracker = ProgressTracker(handler=lambda *a: events.append(a[0]))

    class Thing:
        name = 'thing'
        progress_tracker = tracker

        @track_method('forward')
        def forward(self, x):
            return x + 1
    tracker.register_layer('thing')
    assert Thing().forward(1) == 2
    assert events == ['forward', 'forward']
    summary = tracker.get_summary()['thing'][0]
    assert summary['name'] == 'forward' and summary['done'] and summary['counter'] == 1


# ----------------------------------------------------------------------------- data-parallel host logic

def _char_like_ranges():
    """Flat layout of make_char as nn.flat.FlatParameters builds it: the L2 group (convs) first, then the
    unregularised FullyConnected layers, each group in evaluation order."""
    sizes = [('conv_1', 5 * 3 * 1 * 64 + 64), ('conv_2', 5 * 3 * 64 * 64 + 64), ('conv_3', 5 * 3 * 64 * 64 + 64),
             ('dense_1', 513 * 1024), ('dense_2', 1025 * 128), ('dense_3', 129 * 162)]
    ranges, off = {}, 0
    for name, n in sizes:
        n_al = (n + 3) // 4 * 4
        ranges[name] = (off, off + n_al)
        off += n_al
    return ranges, off


def test_bucket_scheduler_sends_every_gradient_once_largest_layers_first():
    from univer_ocr_b200.nn.flat import BucketScheduler
    ranges, total = _char_like_ranges()
    sched = BucketScheduler(ranges, bucket_elems=(256 << 10) // 4)
    backward_order = ['dense_3', 'leaky_relu_2', 'dense_2', 'leaky_relu_1', 'dense_1', 'flatten', 'fixed_width',
                      'conv_3', 'conv_2', 'conv_1']
    sent, timeline = [], []
    for name in backward_order:
        out = sched.layer_done(name)
        sent += out
        timeline.append((name, out))
    sent += sched.finish()
    covered = sorted(sent)
    assert covered[0][0] == 0 and covered[-1][1] == total
    assert all(a[1] == b[0] for a, b in zip(covered, covered[1:]))           # a partition: no gap, no overlap
    # dense_3 alone (20 898 gradients) stays below the 64 Ki-element threshold and rides with dense_2
    assert timeline[0][1] == [] and timeline[2][1] == [(ranges['dense_2'][0], ranges['dense_3'][1])]
    assert timeline[4][1] == [ranges['dense_1']]                             # 2.1 MB leave as soon as dense_1 is done
    # the conv group is not adjacent to anything pending and conv_1 (1 024 gradients) only leaves at the end
    assert sent[-1][0] == 0
    # a second step starts clean
    sched.reset()
    assert sched.layer_done('dense_1') == [ranges['dense_1']]
    assert sched.layer_done('dense_1') == []                                 # reported twice: sent once


def test_bucket_scheduler_flushes_a_non_adjacent_range_and_unreported_layers():
    from univer_ocr_b200.nn.flat import BucketScheduler
    sched = BucketScheduler({'a': (0, 8), 'b': (8, 16), 'c': (16, 24), 'frozen': (24, 24)}, bucket_elems=1000)
    assert sched.layer_done('c') == []
    assert sched.layer_done('a') == [(16, 24)]                               # not adjacent to c: c leaves, a is pending
    assert sched.layer_done('unknown_activation') == [] and sched.layer_done('frozen') == []
    assert sorted(sched.finish()) == [(0, 8), (8, 16)]                       # pending a + b, which never reported


def test_rendezvous_file_is_unique_per_launch(monkeypatch):
    from univer_ocr_b200 import comm
    a = comm.rendezvous_file({'MASTER_PORT': '29501', 'TORCHELASTIC_RUN_ID': 'none'})
    b = comm.rendezvous_file({'MASTER_PORT': '29502', 'TORCHELASTIC_RUN_ID': 'none'})
    assert a != b and str(os.getppid()) in a                                 # ranks of one launch share their parent
    assert comm.rendezvous_file({'UOCR_RDZV_FILE': '/tmp/x.id'}) == '/tmp/x.id'
    single = comm.init(0, 1)
    assert (single.rank, single.world) == (0, 1) and single.allreduce_host([1.5, 2.0], 'max') == [1.5, 2.0]
    assert single.broadcast_ints([3, 1, 2]) == [3, 1, 2]
    comm.use(None)


def test_package_does_not_import_torch():
    """north_star: no PyTorch in the path.  Nothing under univer_ocr_b200/ may import torch (bench.py's launcher glue
    and the tests are the only users)."""
    import re
    pkg = os.path.join(ROOT, 'univer_ocr_b200')
    offenders = []
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith('.py'):
                text = open(os.path.join(dirpath, f)).read()
                if re.search(r'^\s*(import torch|from torch)', text, re.M):
                    offenders.append(os.path.join(dirpath, f))
    assert offenders == []
