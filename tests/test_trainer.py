"""Epoch driver (SURVEY.md 8f row 1): `univer_ocr_b200.trainer.Trainer` against traces of the
reference's `my_model/trainer.py` on scripted models (tests/golden/trainer_traces.json, generated
by tests/golden/make_trainer_golden.py; compared live as well where UOCR_REFERENCE_ROOT names the reference tree), plus
the batched / sharded behaviour the reference does not have."""
import contextlib
import io
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tests import trainer_cases  # noqa: E402

with open(os.path.join(ROOT, 'tests', 'golden', 'trainer_traces.json')) as fp:
    GOLDEN = json.load(fp)


@pytest.mark.parametrize('scenario', sorted(trainer_cases.SCENARIOS))
def test_trainer_matches_reference_trace(scenario):
    got = trainer_cases.run(scenario, trainer_cases.ours_factory)
    want = GOLDEN[scenario]
    assert got['trace'] == want['trace']                      # sample order, roll-backs, saves, lr at each save
    assert got['best'] == want['best'] and got['best_epoch'] == want['best_epoch']
    assert got['lr'] == want['lr'] and got['weights'] == want['weights']


def test_golden_traces_cover_the_rollback_branches():
    storm = [e for e in GOLDEN['nan_storm']['trace'] if e[0] == 'set_weights']
    assert len(storm) == 11                                   # 9 x last weights, 1 x start weights, 1 x last
    assert storm[9][2] == 0.3                                 # the "too many attempts" branch reloads the START weights
    assert any(e[0] == 'save' for e in GOLDEN['plain']['trace'])


def test_trainer_matches_reference_live():
    """The golden traces against the reference itself.  Without the reference tree, test_trainer_matches_reference_trace
    checks the same scenarios against tests/golden/trainer_traces.json."""
    from oracle import ref_loader
    if not ref_loader.available():
        pytest.skip('reference tree not present')
    ref = ref_loader.load_trainer()
    for scenario in trainer_cases.SCENARIOS:
        with contextlib.redirect_stdout(io.StringIO()):
            want = trainer_cases.run(scenario, trainer_cases.reference_factory(ref))
        assert want == GOLDEN[scenario]
        assert trainer_cases.run(scenario, trainer_cases.ours_factory) == want


def test_losses_table_matches_reference_print():
    from oracle import ref_loader
    if not ref_loader.available():
        pytest.skip('reference tree not present')
    from univer_ocr_b200.trainer import Losses
    ref = ref_loader.load_trainer()
    names, cnts = ['monochrome', 'line'], {'monochrome': 1, 'line': 2}
    tables = []
    for cls in (ref.Losses, Losses):
        l = cls(names, cnts)
        l.reset()
        l.train({'monochrome': {'output_losses': [1.5]}, 'line': {'output_losses': [0.25, 3.0]}})
        l.validation({'monochrome': {'output_losses': [2.5]}, 'line': {'output_losses': [0.125, 1.0]}})
        l.normalize(2, 4)
        l.next()
        l.reset()
        l.train({'monochrome': {'output_losses': [1.0]}, 'line': {'output_losses': [0.5, 2.0]}})
        l.validation({'monochrome': {'output_losses': [2.0]}, 'line': {'output_losses': [0.25, 0.5]}})
        l.normalize(2, 4)
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            l.print(left_margin=2)
        tables.append(buf.getvalue())
    assert tables[0] == tables[1] and 'Avg loss change' in tables[0]


class _MeanModel(trainer_cases.ScriptedModel):
    """A model whose loss averages over the batch (like SoftmaxCE), with a linear update rule so
    that a stacked batch can be compared with per-sample arithmetic."""
    mean_over_batch = True

    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self.seen = []

    def train(self, X, y):
        self.seen.append(X.shape[0])
        return super().train(X, y)


def test_batched_steps_stack_samples_and_weight_mean_losses():
    from univer_ocr_b200.trainer import Trainer
    opt = trainer_cases.ScriptedOptimizer(0.0)                 # lr 0: weights fixed, losses comparable
    model = _MeanModel('m', 0.5, opt)
    train_ds = trainer_cases.ScriptedDataset(['m'], 7, 3)
    val_ds = trainer_cases.ScriptedDataset(['m'], 3, 4)
    t = Trainer({'m': model}, train_ds, val_ds, optimizer=opt, batch_size=4, log=lambda *a, **k: None)
    best, epoch = t.train(1)
    assert model.seen == [4, 3]                                # 7 samples: one full stack, one ragged
    # the model's loss on a stack uses the stack mean of x; weighting by the stack size keeps the
    # epoch sum on the per-sample scale: sum_b n_b * (w - mean_b)^2 / n_val
    xs = [float(np.mean(val_ds.get(i)['m'][0])) for i in range(3)]
    want = 3 * (0.5 - np.mean(xs)) ** 2 / 3
    assert abs(best['m'][0] - want) < 1e-12 and epoch == {'m': 1}


def _two_rank_worker(rank, world, port, out, mode):
    sys.path.insert(0, ROOT)
    import random
    import torch.distributed as dist
    os.environ['MASTER_ADDR'], os.environ['MASTER_PORT'] = '127.0.0.1', str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from tests.gloo_comm import GlooComm
    from univer_ocr_b200.trainer import Trainer
    opt = trainer_cases.ScriptedOptimizer(0.0)
    trace = []
    model = trainer_cases.ScriptedModel('m', 0.5, opt, trace=trace)
    train_ds = trainer_cases.ScriptedDataset(['m'], 7, 3)         # 7 samples, stacks of 2: the last, single sample is dropped
    val_ds = trainer_cases.ScriptedDataset(['m'], 4, 4)
    saves = []
    kwargs = {}
    if mode == 'fixed':
        kwargs['shuffle'] = lambda order: None
    else:                                                         # the default random.shuffle, seeded DIFFERENTLY per rank
        random.seed(1000 + rank)
    t = Trainer({'m': model}, train_ds, val_ds, optimizer=opt, batch_size=2, save_weights_func=saves.append,
                log=lambda *a, **k: None, comm=GlooComm(), **kwargs)
    best, _ = t.train(1)
    out.put((rank, best['m'][0], [e[2] for e in trace if e[0] == 'train'], len(saves)))
    dist.destroy_process_group()


def _run_two_ranks(mode, port_base):
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    out = ctx.Queue()
    port = port_base + os.getpid() % 90
    procs = [ctx.Process(target=_two_rank_worker, args=(r, 2, port, out, mode)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    return sorted(out.get(timeout=10) for _ in range(2))


def test_two_ranks_shard_each_batch_and_agree_on_losses():
    got = _run_two_ranks('fixed', 29900)
    train_ds = trainer_cases.ScriptedDataset(['m'], 7, 3)
    val_ds = trainer_cases.ScriptedDataset(['m'], 4, 4)
    x = [round(float(np.mean(train_ds.get(i)['m'][0])), 9) for i in range(6)]
    assert got[0][2] == x[0:6:2] and got[1][2] == x[1:6:2]     # rank r trains samples r, r + world, ...; both run 3 steps
    want = sum((0.5 - float(np.mean(val_ds.get(i)['m'][0]))) ** 2 for i in range(4)) / 4
    assert abs(got[0][1] - want) < 1e-12 and got[0][1] == got[1][1]   # losses summed over ranks
    assert (got[0][3], got[1][3]) == (1, 0)                    # only rank 0 saves


def test_two_ranks_agree_on_the_shuffled_order():
    """Per-process random.shuffle (differently seeded ranks): rank 0's permutation is broadcast, so the two ranks'
    slices are disjoint and together cover the 6 samples an epoch consumes (7 samples, stacks of 2, world 2)."""
    got = _run_two_ranks('random', 29800)
    train_ds = trainer_cases.ScriptedDataset(['m'], 7, 3)
    x = [round(float(np.mean(train_ds.get(i)['m'][0])), 9) for i in range(7)]
    seen = got[0][2] + got[1][2]
    assert len(got[0][2]) == len(got[1][2]) == 3
    assert len(set(seen)) == 6 and set(seen) <= set(x)         # a partition: nothing trained twice, one sample left out
    assert got[0][1] == got[1][1]


def test_multi_rank_rejects_samples_that_miss_a_model():
    from univer_ocr_b200.trainer import Trainer

    class TwoRanks:
        rank, world = 0, 2

        def allreduce_host(self, values, op='sum'):
            return list(values)

        def broadcast_ints(self, values, root=0):
            return list(values)

    opt = trainer_cases.ScriptedOptimizer(0.0)
    models = {'a': trainer_cases.ScriptedModel('a', 0.5, opt), 'b': trainer_cases.ScriptedModel('b', 0.5, opt)}
    full = trainer_cases.ScriptedDataset(['a', 'b'], 4, 3)

    class Ragged:
        def __len__(self):
            return 4

        def get(self, i):
            sample = full.get(i)
            if i == 2:
                del sample['b']
            return sample

    t = Trainer(models, Ragged(), full, optimizer=opt, batch_size=2, log=lambda *a, **k: None, comm=TwoRanks(),
                shuffle=lambda order: None, prefetch=0)
    with pytest.raises(ValueError, match='every model in every sample'):
        t.train(1)


def test_prefetch_overlaps_host_batching_with_training_and_keeps_order():
    import time
    from univer_ocr_b200.trainer import Trainer

    class SlowDataset(trainer_cases.ScriptedDataset):
        def get(self, i):
            time.sleep(0.01)
            return super().get(i)

    class SlowModel(trainer_cases.ScriptedModel):
        def train(self, X, y):
            time.sleep(0.02)
            return super().train(X, y)

    def run(prefetch):
        opt = trainer_cases.ScriptedOptimizer(0.01)
        trace = []
        model = SlowModel('m', 0.5, opt, trace=trace)
        t = Trainer({'m': model}, SlowDataset(['m'], 16, 3), trainer_cases.ScriptedDataset(['m'], 2, 4), optimizer=opt,
                    batch_size=2, prefetch=prefetch, shuffle=lambda order: order.reverse(), log=lambda *a, **k: None)
        t0 = time.perf_counter()
        best, _ = t.train(1)
        return time.perf_counter() - t0, [e[2] for e in trace if e[0] == 'train'], best

    t_serial, order_serial, best_serial = run(0)
    t_prefetch, order_prefetch, best_prefetch = run(2)
    assert order_prefetch == order_serial and best_prefetch == best_serial      # same batches, same order
    assert t_serial > 0.30 and t_prefetch < t_serial - 0.08                       # 8 x (2 x 10 ms) of fetching hidden


def test_prefetch_propagates_dataset_errors():
    from univer_ocr_b200.trainer import Trainer

    class Broken(trainer_cases.ScriptedDataset):
        def get(self, i):
            if i == 5:
                raise KeyError('sample 5 is missing')
            return super().get(i)

    opt = trainer_cases.ScriptedOptimizer(0.01)
    t = Trainer({'m': trainer_cases.ScriptedModel('m', 0.5, opt)}, Broken(['m'], 8, 3),
                trainer_cases.ScriptedDataset(['m'], 2, 4), optimizer=opt, batch_size=2, shuffle=lambda order: None,
                log=lambda *a, **k: None)
    with pytest.raises(KeyError):
        t.train(1)
