#!/usr/bin/env python
"""Headline benchmark: my_model inference images/s (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One STEP = one pass of the four sub-networks' forward over one batch of synthetic inputs per
GPU (page-sharded, no collective, weak scaling):
    Monochrome -> Paragraph on 64 page tiles (64, 496, 736, 1)
    Line  on 64 line tiles  (64, 128, 256, 1)
    Char  on 64 char lines  (64, 32, 256, 1)  (-> 16384 windows x 162 classes)
`value` = page tiles / s over all GPUs with float32 inputs resident in HBM (CUDA events, max over
ranks).  `e2e` = the same four forward passes through the public pipelined API with pinned HOST buffers,
H2D and D2H inside the timed region, in the forms the reference's neighbouring stages use: 8-bit image
planes in (`train_data_generator.py:24-37`), thresholded uint8 masks and the PredToText hit table out
(`interpreter/interpreter.py:437-447, 596-602`); `e2e.float_out_value` is the all-float32 variant.
Extra keys of the same JSON line: `train` (BASELINE configs[2]: data-parallel training step, weak scaling
at 64 tiles per GPU, and `train.global_512` = global batch 512 as the config is written), `fullpage`
(configs[3]: 64 pages of 2064 x 2064 sharded over the ranks), `stages` (the crop stages between the networks on the
device next to their scipy.ndimage restatement on the host), `roofline`, `cpu_baseline`, `cpu_baseline_train`.
Prints ONE JSON line (rank 0).

`--steps K` is the number of timed steps of `value`, `e2e` (pipelined and synchronous), `train`,
`train.global_512` and `fullpage`; `stages`, `tf32_long_gemm` and the per-layer `layers` breakdown repeat a fixed,
small number of calls.

No PyTorch: ranks rendezvous and reduce through libuocr's own NCCL binding (univer_ocr_b200.comm).

`--impl reference` times the reference's CPU algorithm (oracle port: per-output-pixel NumPy
loops, float64 -- what the reference's `_forward_cpu` / `_backward_cpu` do) on all host cores, one
sample per core; see cpu_baseline.sample in its line.

`--dump-outputs DIR` writes what the last timed step of `value` returned on rank 0 (the Paragraph, Line and Char
predictions) as DIR/<name>.npy in float32, so that two builds can be compared output for output: inputs and weights
are seeded, so the same arguments give the same inputs.  Above 64 MB in all, every array keeps the same fixed, seeded
fraction of its leading-axis rows (tiles for Paragraph and Line, windows for Char), in order.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PAGE_HW, LINE_HW, CHAR_HW = (496, 736), (128, 256), (32, 256)
FULLPAGE_HW = (2064, 2064)            # 2048 x 2048 after make_divisible_by(16, 16) (my_model/model.py:26-34)
METRIC = 'my_model inference images/sec (page tiles through Monochrome->Paragraph + Line + Char forward)'
UNIT = 'images/s'
# scale of the centred ("signed") weights per sub-network: the reference's kaiming_uniform is all-positive
# (nn/initializers.py:22-25) and saturates every output (sigmoid == 1.0: zero data gradient, constant loss); same
# constants as the parity goldens (oracle/np_models.GOLDEN_SCALE)
SIGNED_SCALE = {'monochrome': 5.0, 'paragraph': 5.5, 'line': 3.5, 'char': 2.5}
DUMP_BYTES = 63 * 10**6               # array data of --dump-outputs; with the .npy headers the dump stays below 64 MB


def load_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        p = json.load(open(path))
        return {'hbm_gbs': float(p['hbm_gbs']), 'bf16_tflops': float(p['bf16_tflops']),
                'bf16_tflops_sustained': float(p.get('bf16_tflops_sustained', p['bf16_tflops'])),
                'source': 'measured (MEASURED_PEAKS.json)'}
    except Exception:
        return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0,
                'source': 'fallback (B200_PROFILING.md)'}


# ------------------------------------------------------------------------------ synthetic data

def synth_tiles(rng, n, hw):
    """SURVEY 8d: U[0,1) paper with sparse dark ink: value = 1 - Bernoulli(0.1) * U[0.5, 1)."""
    h, w = hw
    ink = (rng.random((n, h, w, 1), dtype=np.float32) < 0.1)
    x = 1.0 - ink * rng.uniform(0.5, 1.0, size=(n, h, w, 1)).astype(np.float32)
    return np.ascontiguousarray(x, dtype=np.float32)


def synth_tiles_u8(rng, n, hw):
    """The same tiles as 8-bit image planes (what `encode_layers` divides by 255)."""
    return np.ascontiguousarray(np.rint(synth_tiles(rng, n, hw) * 255.0), dtype=np.uint8)


def dump_outputs(directory, outputs, limit=DUMP_BYTES):
    """Writes {name: float32 host array} as <directory>/<name>.npy.  Above `limit` bytes in all, every array keeps the
    same fraction of its leading-axis rows, chosen by a fixed seed and kept in order."""
    os.makedirs(directory, exist_ok=True)
    total = sum(a.nbytes for a in outputs.values())
    for name, a in outputs.items():
        assert a.dtype == np.float32, (name, a.dtype)
        if total > limit:
            keep = max(1, a.shape[0] * limit // total)
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(directory, name + '.npy'), a)


def signed_init(model, scale, with_bias):
    """Centres every weight tensor (and, for the segmentation networks, bias vector) and scales it, on the host."""
    for key, p in model.params().items():
        v = np.asarray(p.value.get(), dtype=np.float64)
        if key.endswith('/w'):
            p.value = (v - v.mean()) * scale
        elif with_bias:
            p.value = (v - v.mean()) * scale if v.size > 1 else v * 0.25


# ------------------------------------------------------------------------------ clocks sampler

class ClockSampler:
    QUERY = ('clocks.sm,clocks.max.sm,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.gpu_index, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.gpu_index), f'--query-gpu={self.QUERY}',
                 '--format=csv,noheader,nounits', '-lms', '100'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in self.lines:
            parts = [p.strip() for p in line.split(',')]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None,
                'sm_max_mhz': float(max(mx)) if mx else None, 'reasons': sorted(reasons),
                'samples': len(sm)}


# ------------------------------------------------------------------------------ B200 arm

class Timer:
    """CUDA-event timing on the compute stream, barrier on both sides, max over ranks."""

    def __init__(self, comm, nn, lib):
        self.comm, self.nn, self.lib = comm, nn, lib

    def event(self):
        e = ctypes.c_void_p()
        self.lib.uocr_event_create(ctypes.byref(e))
        return e.value

    def barrier(self):
        self.comm.barrier()
        self.nn.CP.synchronize()

    def device_ms(self, fn, steps):
        """-> (ms per step, max over ranks; kernel launches of this rank)."""
        from univer_ocr_b200._lib import launch_count
        stream = self.nn.CP.stream()
        self.nn.CP.synchronize()
        self.barrier()
        e0, e1 = self.event(), self.event()
        launches0 = launch_count()
        self.lib.uocr_event_record(e0, stream)
        for i in range(steps):
            fn(i)
        self.lib.uocr_event_record(e1, stream)
        self.lib.uocr_event_sync(e1)
        self.nn.CP.synchronize()
        launches = launch_count() - launches0
        self.barrier()
        ms = ctypes.c_float(0)
        self.lib.uocr_event_elapsed_ms(e0, e1, ctypes.byref(ms))
        return self.comm.allreduce_host([ms.value / steps], 'max')[0], int(launches)

    def wall_s(self, fn, steps):
        """Host wall clock per step of `fn(i)` (the end-to-end legs end with results on the host), max over ranks."""
        self.barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            fn(i)
        dt = (time.perf_counter() - t0) / steps
        return self.comm.allreduce_host([dt], 'max')[0]


def run_b200(args):
    os.environ.setdefault('UOCR_DEVICE', os.environ.get('LOCAL_RANK', '0'))
    import univer_ocr_b200.nn as nn
    from univer_ocr_b200 import comm as comm_, glue, my_model, roofline
    from univer_ocr_b200._lib import lib
    from univer_ocr_b200.nn.progress_tracker import BaseProgressTracker, CudaEventTracker
    from univer_ocr_b200.pipeline import CapturedStep, ConcurrentBranches, InferencePipeline

    nn.CP.use_gpu()
    nn.CP.set_math_mode(args.math)
    comm = comm_.init_from_env()
    timer = Timer(comm, nn, lib)
    B = args.batch
    rng = np.random.default_rng(1234 + comm.rank)
    np.random.seed(1234)                                # layer initialisers draw from np.random: same weights on every rank
    train_opt = nn.optimizers.Adam(lr=0.0015)           # one Adam instance shared by the four networks (my_model/train.py:127)
    models = {
        'monochrome': my_model.make_monochrome((B, *PAGE_HW, 1), optimizer=train_opt),
        'paragraph': my_model.make_paragraph((B, *PAGE_HW, 1), optimizer=train_opt),
        'line': my_model.make_line((B, *LINE_HW, 1), optimizer=train_opt),
        'char': my_model.make_char((B, *CHAR_HW, 1), optimizer=train_opt),
    }
    for name, model in models.items():                  # signed weights: outputs spread over (0, 1), losses move
        signed_init(model, SIGNED_SCALE[name], with_bias=name != 'char')

    n_sets = 2                                           # rotate inputs: 2 x 103 MB > L2, plus
    host_sets, host_sets_u8 = [], []                     # ~3.3 GB of intermediates per step
    for _ in range(n_sets):
        hs, hs8 = {}, {}
        for key, hw in (('page', PAGE_HW), ('line', LINE_HW), ('char', CHAR_HW)):
            u8 = synth_tiles_u8(rng, B, hw)
            buf8 = nn.CP.pinned_empty(u8.shape, np.uint8)
            buf8[...] = u8
            buf = nn.CP.pinned_empty(u8.shape, np.float32)
            buf[...] = (u8 / 255.0).astype(np.float32)   # the float32 storage of the reference's float64 u / 255
            hs[key], hs8[key] = buf, buf8
        host_sets.append(hs)
        host_sets_u8.append(hs8)
    dev_sets = [{k: nn.CP.copy(np.asarray(v)) for k, v in hs.items()} for hs in host_sets]
    nn.CP.synchronize()

    # the Monochrome -> Paragraph chain, Line and Char do not feed each other: three forked streams, joined on the
    # compute stream (UOCR_BENCH_SERIAL=1: one stream, e.g. for per-layer timing)
    fork = None if os.environ.get('UOCR_BENCH_SERIAL') == '1' else ConcurrentBranches(3)

    def step_serial(inp):
        mono = models['monochrome'].predict(inp['page'])[0]
        para = models['paragraph'].predict(mono)[0]
        line = models['line'].predict(inp['line'])[0]
        char = models['char'].predict(inp['char'])[0]
        return para, line, char

    def eager_step(inp):
        if fork is None:
            return step_serial(inp)
        return tuple(fork.run(lambda: models['paragraph'].predict(models['monochrome'].predict(inp['page'])[0])[0],
                              lambda: models['line'].predict(inp['line'])[0],
                              lambda: models['char'].predict(inp['char'])[0]))

    def e2e_step(inp_u8):
        """uint8 planes in -> the forms the next host stages consume out: binarised paragraph / line masks
        (interpreter.py:437-447) and the PredToText hit table (:596-602)."""
        def page_branch():
            x = glue.pixels_to_unit(inp_u8['page'])
            return glue.thresholded(models['paragraph'].predict(models['monochrome'].predict(x)[0])[0])

        def line_branch():
            return glue.thresholded(models['line'].predict(glue.pixels_to_unit(inp_u8['line']))[0])

        def char_branch():
            return glue.row_max_hits(models['char'].predict(glue.pixels_to_unit(inp_u8['char']))[0])
        if fork is None:
            return page_branch(), line_branch(), char_branch()
        return tuple(fork.run(page_branch, line_branch, char_branch))

    # ---------------- device-resident throughput (`value`) ----------------
    # the step over a resident input set is a fixed launch sequence: captured once per set into a CUDA graph
    # (pipeline.CapturedStep; UOCR_BENCH_GRAPH=0 issues the launches one by one instead)
    use_graph = os.environ.get('UOCR_BENCH_GRAPH', '1') != '0'
    graph_note = None
    step = eager_step
    if use_graph:
        captured = {id(inp): CapturedStep(lambda inp=inp: eager_step(inp)) for inp in dev_sets}
        try:                                             # capture now; a failure falls back to eager launches, loudly
            for graph in captured.values():
                graph()
            nn.CP.synchronize()

            def step(inp):
                return captured[id(inp)]()
        except Exception as exc:                         # noqa: BLE001
            graph_note = f'graph capture failed, launching kernel by kernel: {exc}'
            print(graph_note, file=sys.stderr, flush=True)
            use_graph = False

    for i in range(max(args.warmup, n_sets)):
        step(dev_sets[i % n_sets])
    sampler = ClockSampler(int(os.environ.get('LOCAL_RANK', '0')))
    sampler.start()
    last = []

    def timed_step(i):
        out = step(dev_sets[i % n_sets])
        if i == args.steps - 1:
            last.append(out)
    ms_per_step, launches = timer.device_ms(timed_step, args.steps)
    value = B * comm.world / (ms_per_step / 1e3)
    if args.dump_outputs and comm.rank == 0:
        dump_outputs(args.dump_outputs, {name: o.get() for name, o in zip(('paragraph', 'line', 'char'), last[0])})
    del last

    # ---------------- end to end through the public API with host buffers (`e2e`) ----------------
    # the pipelined public API (univer_ocr_b200.pipeline.InferencePipeline): H2D of batch i+1, forward of batch i and
    # D2H of batch i-1 overlap on three streams; every batch is uploaded from and downloaded to pinned host memory
    # inside the timed region.  The untimed warm-up batches leave the pipeline full (as W warm-up steps leave a model
    # warm): the region runs from the submission of the first timed batch to the retirement of the LAST timed batch, so
    # it contains the upload, the forward and the download of each of the K timed batches (plus the downloads of the
    # warm-up batches still in flight when it starts) -- the final drain is inside, the initial fill is not.
    e2e_depth = int(os.environ.get('UOCR_BENCH_DEPTH', '3'))

    def pipelined(fn, sets):
        pipe = InferencePipeline(fn, depth=e2e_depth, graph=use_graph)
        for i in range(6):
            pipe.submit(sets[i % n_sets], i)
        outs = [o for _, o in pipe.drain()][-1]
        warm = max(args.warmup, 2 * e2e_depth)
        for i in range(warm):                                # refill: these batches are in flight when the clock starts
            pipe.submit(sets[i % n_sets], ('warm', i))
        timed = [0]

        def count(done):
            if done is not None and done[0][0] == 'timed':
                timed[0] += 1
        timer.barrier()
        t0 = time.perf_counter()
        for i in range(args.steps):
            count(pipe.submit(sets[i % n_sets], ('timed', i)))
        for done in pipe.drain():
            count(done)
        sec = comm.allreduce_host([(time.perf_counter() - t0) / args.steps], 'max')[0]
        assert timed[0] == args.steps
        return sec, sum(v.nbytes for v in sets[0].values()), sum(o.nbytes for o in outs)

    e2e_s, h2d, d2h = pipelined(e2e_step, host_sets_u8)
    f32_s, f32_h2d, f32_d2h = pipelined(eager_step, host_sets)
    # synchronous form of the same call: upload, forward, download, wait -- one batch at a time
    sync_host = None

    def e2e_sync(i):
        nonlocal sync_host
        inp = {k: nn.DeviceArray.from_host(v, np.uint8) for k, v in host_sets_u8[i % n_sets].items()}
        outs = e2e_step(inp)
        if sync_host is None:
            sync_host = [nn.CP.pinned_empty(o.shape, o.dtype) for o in outs]
        for o, h in zip(outs, sync_host):
            lib.uocr_memcpy_d2h(h.ctypes.data, o.ptr, o.nbytes, nn.CP.stream())
        nn.CP.synchronize()
    for i in range(3):
        e2e_sync(i)
    timer.barrier()
    sync_times = []
    for i in range(args.steps):
        t0 = time.perf_counter()
        e2e_sync(i)
        sync_times.append(time.perf_counter() - t0)
    # median per call: an occasional host hiccup (allocator, Python GC) of tens of ms would otherwise dominate a 10-call mean
    sync_s = comm.allreduce_host([float(np.median(sync_times))], 'max')[0]
    clocks = sampler.stop()

    # ---------------- per-layer device time -> dominant kernel -> roofline ----------------
    peaks = load_peaks()
    in_shapes = {'monochrome': (B, *PAGE_HW, 1), 'paragraph': (B, *PAGE_HW, 1),
                 'line': (B, *LINE_HW, 1), 'char': (B, *CHAR_HW, 1)}
    for i in range(2):                                           # the serial order allocates from the compute stream's
        step_serial(dev_sets[i % n_sets])                        # pool: fill it before timing layers
    nn.CP.synchronize()
    tracker = CudaEventTracker()
    work = {}
    for mname, model in models.items():
        work.update(roofline.plan_work(model, in_shapes[mname], training=False))
        for layer in model.layers.values():
            layer.progress_tracker = tracker
    prof_steps = max(2, min(args.steps, 5))
    for i in range(prof_steps):
        step_serial(dev_sets[i % n_sets])                      # per-layer event pairs: one stream
    per_layer = tracker.summary_ms()
    for model in models.values():
        for layer in model.layers.values():
            layer.progress_tracker = BaseProgressTracker()
    total_ms = sum(v[0] for v in per_layer.values()) / prof_steps
    breakdown = sorted(((name, v[0] / v[1]) for (name, ev), v in per_layer.items() if ev == 'forward'),
                       key=lambda t: -t[1])
    top_name, top_ms = breakdown[0]
    wk = work[top_name]
    tf32_peak = peaks['bf16_tflops'] / 2.0
    if wk['bound'] == 'tensor':
        achieved = wk['flops'] / (top_ms / 1e3) / 1e12
        roof = {'bound': 'tensor', 'achieved': achieved, 'peak': tf32_peak, 'unit': 'TFLOP/s',
                'frac': achieved / tf32_peak, 'traffic': None,
                'peak_note': f'TF32 dense taken as 1/2 of bf16 burst {peaks["bf16_tflops"]} TF/s, {peaks["source"]}'}
    else:
        achieved = wk['bytes'] / (top_ms / 1e3) / 1e9
        roof = {'bound': 'hbm', 'achieved': achieved, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
                'frac': achieved / peaks['hbm_gbs'], 'traffic': None, 'peak_note': peaks['source']}
    try:                                            # DRAM traffic of that kernel from the committed ncu capture
        tr = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json'))).get('+'.join(wk.get('fused', [top_name])))
        if tr and tr['batch'] == B:
            roof['traffic'] = tr['bytes']
            roof['traffic_source'] = tr['profile']
            if tr.get('note'):
                roof['note'] = tr['note']
    except (OSError, ValueError):
        pass
    roof.update({'kernel': '+'.join(wk.get('fused', [top_name])), 'kernel_ms': top_ms, 'share_of_step': top_ms / total_ms,
                 'algorithmic_bytes': wk['bytes'], 'algorithmic_flops': wk['flops']})
    layers_out = []
    for name, lms in breakdown[:12]:
        w_ = work[name]
        layers_out.append({'layer': '+'.join(w_.get('fused', [name])), 'ms': round(lms, 4), 'bound': w_['bound'],
                           'GBps': round(w_['bytes'] / (lms / 1e3) / 1e9, 1),
                           'TFLOPs': round(w_['flops'] / (lms / 1e3) / 1e12, 2),
                           'frac_of_roof': round((w_['flops'] / (lms / 1e3) / 1e12 / tf32_peak) if w_['bound'] == 'tensor'
                                                 else (w_['bytes'] / (lms / 1e3) / 1e9 / peaks['hbm_gbs']), 3)})
    tf32_measured = None
    if comm.rank == 0 and not args.no_gemm_peak:
        tf32_measured = measure_long_gemm(nn, lib, timer)

    train = None if args.no_train else measure_train(args, comm, timer, nn, my_model, models, dev_sets, rng, B)
    fullpage = None if args.no_fullpage else measure_fullpage(args, comm, timer, nn, my_model, rng)

    result = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': comm.world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32' if args.math == 'fp32' else 'tf32/f32',
        'data': 'synthetic',
        'config': {'workload': 'BASELINE configs[1]: my_model inference, batch 64 synthetic page tiles '
                               '(64,496,736,1) Monochrome->Paragraph + Line (64,128,256,1) + Char '
                               '(64,32,256,1), per GPU; pages sharded across GPUs, no collective',
                   'batch_per_gpu': B, 'math_mode': args.math,
                   'weights': 'kaiming_uniform draws (seeded), centred and scaled per network so that outputs are not saturated',
                   'streams': 'Monochrome->Paragraph, Line and Char forward on three forked CUDA streams joined per step' if fork is not None else 'one stream',
                   'launch': 'one CUDA graph replay per step (captured per resident input set)' if use_graph else (graph_note or 'kernel by kernel'),
                   'collectives': 'libuocr NCCL binding (univer_ocr_b200.comm), no PyTorch; NCCL %s' % (comm_.Communicator.version() if comm.world > 1 else 'not loaded'),
                   'l2_policy': 'inputs rotate over 2 resident sets (206 MB) and each step streams '
                                '~3.3 GB of intermediates: working set >> 126 MB L2'},
        'e2e': {'value': B * comm.world / e2e_s, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                'ms_per_step': e2e_s * 1e3,
                'api': 'univer_ocr_b200.pipeline.InferencePipeline(depth=%d%s): pinned host uint8 planes -> H2D -> /255 on the device -> four forward passes -> thresholded uint8 masks (paragraph, line) + PredToText uint8 hit table (char) -> D2H -> pinned host' % (e2e_depth, ', graph=True' if use_graph else ''),
                'timing': 'host wall clock from the submission of the first timed batch to the retirement of the last one (K batches: each one\'s H2D, forward and D2H inside; the untimed warm-up batches keep the pipeline full at the start, the final drain is inside), max over ranks',
                'sync_value': B * comm.world / sync_s, 'sync_ms_per_step': sync_s * 1e3,
                'sync_timing': 'median host wall clock of one synchronous call (upload, forward, download, wait)',
                'float_out_value': B * comm.world / f32_s, 'float_out_ms_per_step': f32_s * 1e3,
                'float_out_h2d_bytes_per_step': f32_h2d, 'float_out_d2h_bytes_per_step': f32_d2h},
        'gpu_launches': int(launches),
        'clocks': clocks,
        'roofline': roof,
        'layers': layers_out,
    }
    if tf32_measured is not None:
        result['tf32_long_gemm'] = tf32_measured
    if train is not None:
        result['train'] = train
    if fullpage is not None:
        result['fullpage'] = fullpage
    if comm.rank == 0 and not args.no_stages:
        result['stages'] = measure_stages(nn, lib)
    if comm.rank == 0 and comm.world == 1 and not args.no_cpu_baseline:
        result['cpu_baseline'] = cpu_baseline(budget_s=args.cpu_budget, cores=1)
        result['cpu_baseline_train'] = cpu_baseline(budget_s=args.cpu_budget, cores=1, train=True)
    if comm.rank == 0:
        print(json.dumps(result), flush=True)
    comm.close()


def measure_stages(nn, lib):
    """SURVEY 8f row 4: the crop stages between the sub-networks (interpreter.py:234-523) on one synthetic page tile with
    two tilted paragraphs and on two cropped paragraphs of three lines each -- device classes (univer_ocr_b200.stages,
    results stay on the device; the timed region ends with a device synchronise) next to the CPU restatement with
    scipy.ndimage (oracle/np_stages.py, single process; the reference spreads the same calls over worker processes).
    Host wall clock: the stages are host-driven object loops around small kernels."""
    import time
    from oracle import np_stages
    from tests import stage_cases
    from univer_ocr_b200 import stages
    from univer_ocr_b200._lib import launch_count
    pred, images = stage_cases.paragraph_page(0, h=PAGE_HW[0], w=PAGE_HW[1])
    images = images[:1]                                        # PREDICT mode cuts the Monochrome map only
    lines = [stage_cases.line_paragraph(s, None, h=128, w=512, lines=3) for s in (1, 2)]
    masks, arrays = [m for m, _ in lines], [[a[0] for _, a in lines]]
    d_pred, d_images = nn.CP.copy(pred), [nn.CP.copy(i) for i in images]
    d_masks, d_arrays = [nn.CP.copy(m) for m in masks], [[nn.CP.copy(a) for a in arrays[0]]]
    para = stages.CropAndRotateParagraphs(None, True)
    line = stages.CropRotateAndZoomLines(None, 32, 8)

    def device_pass():
        para(d_pred, d_images)
        line(d_masks, d_arrays)
        nn.CP.synchronize()
    device_pass()
    n0, reps = launch_count(), 5
    t0 = time.perf_counter()
    for _ in range(reps):
        device_pass()
    dev_s = (time.perf_counter() - t0) / reps
    launches = (launch_count() - n0) // reps
    t0 = time.perf_counter()
    want_p, angles = np_stages.crop_and_rotate_paragraphs(pred, images, True)
    want_l = np_stages.crop_rotate_and_zoom_lines(masks, arrays, 32, 8)
    cpu_s = time.perf_counter() - t0
    got_p = stages.CropAndRotateParagraphs(None, True, to_host=True)(d_pred, d_images)
    got_l = stages.CropRotateAndZoomLines(None, 32, 8, to_host=True)(d_masks, d_arrays)
    same = (all(np.array_equal(g, w) for g, w in zip(got_p[0], want_p[0]))
            and all(np.array_equal(g, w) for gp, wp in zip(got_l[0], want_l[0]) for g, w in zip(gp, wp)))
    return {'metric': 'crop stages per page tile: CropAndRotateParagraphs (rotation search on) + CropRotateAndZoomLines',
            'workload': '1 page tile %dx%d with 2 tilted paragraphs (1 map cut) + 2 paragraphs 128x512 with 3 lines each, '
                        'zoomed to height 32' % PAGE_HW,
            'device_ms': dev_s * 1e3, 'cpu_ms': cpu_s * 1e3, 'cpu_kind': 'port (scipy.ndimage, 1 process)',
            'gpu_launches': int(launches), 'angles': angles, 'bit_identical_to_cpu': bool(same)}


def measure_long_gemm(nn, lib, timer):
    """SURVEY 8d: 'TF32 ~ 1/2 of BF16 -- measure, don't assume'.  The repo's own persistent tcgen05 GEMM on a long
    problem (65536 x 1024 x 1024, operands 536 MB >> L2) is the best TF32 rate this code base has demonstrated on the
    box; reported next to the 1/2-of-BF16 proxy the roofline fractions use (the proxy stays the denominator: a peak
    measured with one's own kernel can only flatter)."""
    from univer_ocr_b200._lib import ACT_NONE, MATH_TF32
    M, K, N = 65536, 1024, 1024
    rng = np.random.default_rng(0)
    X = nn.CP.copy(rng.standard_normal((M, K), dtype=np.float32))
    W = nn.CP.copy((rng.standard_normal((K + 1, N), dtype=np.float32) / np.float32(np.sqrt(K))))
    wt, y = nn.DeviceArray((N, K)), nn.DeviceArray((M, N))
    st = nn.CP.stream()
    lib.uocr_weights_to_kmajor(W.ptr, wt.ptr, K, N, st)

    def run(_):
        lib.uocr_fc_fwd_kmajor(X.ptr, W.ptr, wt.ptr, y.ptr, M, K, N, ACT_NONE, 0.0, MATH_TF32, nn.CP.stream())
    for i in range(3):
        run(i)
    nn.CP.synchronize()
    e0, e1 = timer.event(), timer.event()
    reps = 20
    lib.uocr_event_record(e0, st)
    for i in range(reps):
        run(i)
    lib.uocr_event_record(e1, st)
    lib.uocr_event_sync(e1)
    ms = ctypes.c_float(0)
    lib.uocr_event_elapsed_ms(e0, e1, ctypes.byref(ms))
    t = ms.value / reps / 1e3
    return {'shape_mkn': [M, K, N], 'ms': t * 1e3, 'tflops': 2.0 * M * K * N / t / 1e12,
            'kernel': 'tc_gemm_persistent_kernel (uocr_fc_fwd_kmajor, TF32 operands, FP32 accumulate)'}


def make_targets(nn, my_model, rng, B):
    t = {
        'monochrome': nn.CP.copy((rng.random((B, *PAGE_HW, 1), dtype=np.float32) < 0.2).astype(np.float32)),
        'paragraph': nn.CP.copy((rng.random((B, *PAGE_HW, 1), dtype=np.float32) < 0.2).astype(np.float32)),
        'line': nn.CP.copy((rng.random((B, *LINE_HW, 2), dtype=np.float32) < 0.2).astype(np.float32)),
    }
    onehot = np.zeros((B * CHAR_HW[1], my_model.N_CHARS), dtype=np.float32)
    onehot[np.arange(onehot.shape[0]), rng.integers(0, my_model.N_CHARS, size=onehot.shape[0])] = 1
    t['char'] = nn.CP.copy(onehot)
    return t


def measure_train(args, comm, timer, nn, my_model, models, dev_sets, rng, B):
    """BASELINE configs[2]: one data-parallel training step of the four sub-networks (forward + loss + backward +
    bucketed NCCL gradient allreduce overlapped with backward + fused L2/Adam).  Weak scaling at B tiles per GPU, plus
    the config as written (`global_512`: global batch 512, i.e. 512 / world tiles per GPU).  At world > 1 the sharded
    step is first CHECKED against rank 0's full-batch step (`dp_max_rel_err`)."""
    from univer_ocr_b200.parallel import DataParallel
    from univer_ocr_b200.pipeline import CapturedStep, ConcurrentBranches
    out = {}
    if comm.world > 1:
        out['dp_max_rel_err'] = dp_self_check(comm, nn, my_model)
        if not out['dp_max_rel_err'] <= 2e-4:
            raise SystemExit(f'data-parallel self-check failed: max rel err {out["dp_max_rel_err"]:.3e} > 2e-4')

    def build(batch, nets, feeds):
        opt = next(iter(nets['char'].params().values())).optimizer     # the Adam instance the networks were built with
        # Char first: its FullyConnected gradients are 99 % of the bytes on the wire
        order = [n for n in ('char', 'monochrome', 'paragraph', 'line') if n in nets]
        dps = {name: DataParallel(nets[name], optimizer=opt, comm=comm) for name in order}
        targets = make_targets(nn, my_model, rng, batch)
        fork = None if os.environ.get('UOCR_BENCH_SERIAL') == '1' else ConcurrentBranches(len(dps))

        def step(_=None):
            if fork is None:
                return {name: dps[name].train(feeds[name], targets[name]) for name in order}
            outs = fork.run(*[(lambda name=name: dps[name].train(feeds[name], targets[name])) for name in order])
            return dict(zip(order, outs))
        return dps, step

    def timed(step, steps, batch, dps):
        for _ in range(3):
            losses = step()
        nn.CP.synchronize()
        # the training step is a fixed launch sequence over fixed buffers (parameters, gradients and Adam state are
        # updated in place; the NCCL allreduces are captured with it): replayed as ONE CUDA graph unless
        # UOCR_BENCH_TRAIN_GRAPH=0
        launch_mode, run = 'kernel by kernel', step
        if os.environ.get('UOCR_BENCH_TRAIN_GRAPH', '1') != '0':
            def bump():
                nn.CP.weights_generation += 1
            graph = CapturedStep(step, warmup=0, track_weights=False, after_replay=bump)
            try:
                graph()
                nn.CP.synchronize()
                run, launch_mode = (lambda _=None: graph()), 'one CUDA graph replay per step (NCCL allreduces captured)'
            except Exception as exc:                     # noqa: BLE001
                print(f'train-step graph capture failed, launching kernel by kernel: {exc}', file=sys.stderr, flush=True)
        def read(losses):                                # peek: a replayed graph returns the SAME LazyScalar objects
            return {k: v['output_losses'][0].peek() for k, v in losses.items()}
        first = read(run())
        ms, launches = timer.device_ms(run, steps)
        last = read(run())
        n_params = sum(dp.flat.total for dp in dps.values())
        buckets = {name: [hi - lo for lo, hi in dp.buckets_last_step] for name, dp in dps.items()}
        return {'value': batch * comm.world / (ms / 1e3), 'unit': UNIT, 'ms_per_step': ms, 'steps': steps,
                'batch_per_gpu': batch, 'global_batch': batch * comm.world,
                'allreduce_bytes_per_step': 4 * n_params if comm.world > 1 else 0,
                'allreduce_buckets_elems': buckets if comm.world > 1 else {},
                'gpu_launches': launches, 'launch': launch_mode,
                'losses_first_timed_step': first, 'losses_after': last}

    steps = args.steps
    feeds = {'monochrome': dev_sets[0]['page'], 'paragraph': dev_sets[0]['page'], 'line': dev_sets[0]['line'],
             'char': dev_sets[0]['char']}
    dps, step = build(B, models, feeds)
    out.update({'metric': 'my_model train-step images/sec (fwd + loss + bwd + overlapped NCCL grad allreduce + L2 + '
                          'Adam of all four sub-networks)', 'scaling': 'weak'})
    out.update(timed(step, steps, B, dps))
    del dps, step

    if not args.no_global512 and 512 % comm.world == 0:
        # BASELINE configs[2] as written: GLOBAL batch 512 -> 512 / world tiles per GPU (strong scaling over N)
        per = 512 // comm.world
        if per == B:
            out['global_512'] = {k: out[k] for k in ('value', 'ms_per_step', 'batch_per_gpu', 'global_batch', 'steps')}
            out['global_512']['scaling'] = 'strong'
        else:
            np.random.seed(1234)
            opt512 = nn.optimizers.Adam(lr=0.0015)
            nets = {'monochrome': my_model.make_monochrome((per, *PAGE_HW, 1), optimizer=opt512),
                    'paragraph': my_model.make_paragraph((per, *PAGE_HW, 1), optimizer=opt512),
                    'line': my_model.make_line((per, *LINE_HW, 1), optimizer=opt512),
                    'char': my_model.make_char((per, *CHAR_HW, 1), optimizer=opt512)}
            for name, model in nets.items():
                signed_init(model, SIGNED_SCALE[name], with_bias=name != 'char')
            pages = nn.CP.copy(synth_tiles(rng, per, PAGE_HW))
            big = {'monochrome': pages, 'paragraph': pages, 'line': nn.CP.copy(synth_tiles(rng, per, LINE_HW)),
                   'char': nn.CP.copy(synth_tiles(rng, per, CHAR_HW))}
            dps, step = build(per, nets, big)
            # K steps of batch 512 per GPU: at one GPU this section takes about K / 5 times as long as the five steps
            # it once timed regardless of K
            res = timed(step, steps, per, dps)
            res['scaling'] = 'strong'
            out['global_512'] = res
            del dps, step, nets, big, pages
            lib_trim()
    return out


def lib_trim():
    from univer_ocr_b200._lib import lib
    lib.uocr_mempool_trim()


def dp_self_check(comm, nn, my_model):
    """Sharded data-parallel step == full-batch single-process step (FP32 check mode, small shapes).  Every rank trains
    its slice of a batch through `DataParallel` (bucketed allreduce on the side stream) for two steps; before each
    step the full batch goes through a single-process replica holding the SAME weights (forward + loss + backward of
    the per-parameter route, no flat buffers, no collective).  Compared per parameter tensor: the allreduced, scaled
    gradient against the full-batch gradient (max |diff| / max |full|), and the loss (shard losses summed for Dice,
    averaged for SoftmaxCE).  Gradients, not updated weights: Adam without bias correction turns the sign of a
    gradient that is within summation-order rounding of zero into a 2 * 3.16 lr weight difference.
    Returns the maximum over tensors, steps, sub-networks and ranks.  Reference semantics: nn/models.py:232-254,
    nn/losses.py:9-25,60-73."""
    from univer_ocr_b200.parallel import DataParallel
    keep = nn.CP.math_mode
    nn.CP.set_math_mode('fp32')
    world, rank = comm.world, comm.rank
    worst = 0.0
    try:
        for name, shape in (('monochrome', (2 * world, 32, 48, 1)), ('paragraph', (2 * world, 32, 48, 1)),
                            ('line', (2 * world, 32, 64, 1)), ('char', (2 * world, 32, 24, 1))):
            rng = np.random.default_rng(3)                   # the same data on every rank
            X = rng.uniform(size=shape).astype(np.float32)
            np.random.seed(7 + rank)                         # DIFFERENT initial weights per rank: the broadcast must fix it
            local = (shape[0] // world, *shape[1:])
            model = my_model.MAKERS[name](local, optimizer=nn.optimizers.Adam(lr=0.002))
            signed_init(model, SIGNED_SCALE[name], with_bias=name != 'char')
            rows = model.get_output_shapes([local])[0]
            full_rows = (rows[0] * world, *rows[1:])
            if name == 'char':
                y = np.zeros(full_rows, dtype=np.float32)
                y[np.arange(full_rows[0]), rng.integers(0, full_rows[1], full_rows[0])] = 1
            else:
                y = (rng.uniform(size=full_rows) < 0.3).astype(np.float32)
            per_x, per_y = shape[0] // world, full_rows[0] // world
            dp = DataParallel(model, comm=comm, bucket_bytes=4096)    # small buckets: several allreduces per step
            ref = my_model.MAKERS[name](shape, optimizer=nn.optimizers.Adam(lr=0.002))
            ref.fused_update = False
            reduced = {}

            def grab():
                for k, p in model.params().items():
                    reduced[k] = p.grad.get().astype(np.float64) * dp.grad_scale
            dp.after_reduce = grab
            for _ in range(2):
                for k, p in ref.params().items():            # the replica takes the sharded model's current weights
                    p.value = model.params()[k].value.get()
                predicted = ref.forward([X])
                ref_loss, g = ref._loss_for(0)(predicted[0], y)
                ref.backward([g])
                want = {k: p.grad.get().astype(np.float64) for k, p in ref.params().items()}
                out = dp.train(X[rank * per_x:(rank + 1) * per_x], y[rank * per_y:(rank + 1) * per_y])
                for k in want:
                    worst = max(worst, float(np.max(np.abs(reduced[k] - want[k])) / max(float(np.max(np.abs(want[k]))), 1e-30)))
                loss_sum = comm.allreduce_host([float(out['output_losses'][0])], 'sum')[0]
                loss_all = loss_sum * (1.0 if dp.grad_scale == 1.0 else 1.0 / world)
                worst = max(worst, abs(loss_all - float(ref_loss)) / max(abs(float(ref_loss)), 1e-30))
            assert len(dp.buckets_last_step) >= (3 if name == 'char' else 1)      # Char: FC buckets leave before the convs'
    finally:
        nn.CP.math_mode = keep
    return comm.allreduce_host([worst], 'max')[0]


def measure_fullpage(args, comm, timer, nn, my_model, rng):
    """BASELINE configs[3]: 64 full pages (2048 x 2048 -> 2064 x 2064 after make_divisible_by) through
    Monochrome -> Paragraph, pages sharded round-robin over the ranks, no collective (reference path:
    my_model/model.py:26-34, 688-699).  Pages/s from device time, max over ranks."""
    pages, per_launch = 64, 4
    mine = len(range(comm.rank, pages, comm.world))
    launches_per_pass = -(-mine // per_launch)
    shape = (per_launch, *FULLPAGE_HW, 1)
    np.random.seed(1234)
    mono, para = my_model.make_monochrome(shape), my_model.make_paragraph(shape)
    signed_init(mono, SIGNED_SCALE['monochrome'], True)
    signed_init(para, SIGNED_SCALE['paragraph'], True)
    sets = [nn.CP.copy(synth_tiles(rng, per_launch, FULLPAGE_HW)) for _ in range(2)]     # 2 x 68 MB > L2

    def one_pass(_=None):
        for j in range(launches_per_pass):
            para.predict(mono.predict(sets[j % 2])[0])
    for _ in range(2):
        one_pass()
    ms, launches = timer.device_ms(one_pass, args.steps)
    done = launches_per_pass * per_launch * comm.world
    return {'metric': 'full-page inference pages/sec (2064x2064 after make_divisible_by, Monochrome->Paragraph)',
            'value': done / (ms / 1e3), 'unit': 'pages/s', 'pages_per_pass': done, 'pages_per_launch': per_launch,
            'ms_per_pass': ms, 'passes_timed': args.steps, 'gpu_launches': launches, 'scaling': 'strong (64 pages over N GPUs)',
            'l2_policy': 'two resident 4-page input sets (2 x 68 MB) alternate; 273 MB of intermediates per launch'}


# ------------------------------------------------------------------------------ CPU arms
# (the only place outside tests/ and smoke() that executes oracle/)

def _cpu_sample(frac, seed=1234, train=False):
    """Forward (or one whole `Model.train` step: forward + loss + backward + L2 + Adam, reference
    nn/models.py:250-254) of the four sub-networks over a strip of ONE image each with the loop-form oracle port;
    returns seconds.  `frac` = fraction of each tile's rows (columns for Char) processed."""
    from oracle import np_models
    rng = np.random.default_rng(seed)
    rows_p = max(16, int(round(PAGE_HW[0] * frac / 16)) * 16)
    rows_l = max(4, int(round(LINE_HW[0] * frac / 4)) * 4)
    cols_c = max(8, int(round(CHAR_HW[1] * frac)))

    def run(name, x):
        spec, kind = np_models.net_spec(name), np_models.loss_kind(name)
        w = np_models.golden_weights(name, seed)
        if not train:
            return np_models.forward(spec, w, x, loop=True)
        pred = np_models.forward(spec, w, x)                       # vectorised, only to size the target (untimed)
        if kind == 'dice':
            y = (rng.uniform(size=pred.shape) < 0.2).astype(np.float64)
        else:
            y = np.zeros(pred.shape)
            y[np.arange(y.shape[0]), rng.integers(0, y.shape[1], size=y.shape[0])] = 1
        t = time.perf_counter()
        np_models.train_step(spec, kind, w, np_models.new_adam_state(w), x, y, lr=0.0015, loop=True)
        return time.perf_counter() - t

    page = synth_tiles(rng, 1, (rows_p, PAGE_HW[1])).astype(np.float64)
    line = synth_tiles(rng, 1, (rows_l, LINE_HW[1])).astype(np.float64)
    char = synth_tiles(rng, 1, (CHAR_HW[0], cols_c)).astype(np.float64)
    t0 = time.perf_counter()
    if train:
        dt = run('monochrome', page) + run('paragraph', page) + run('line', line) + run('char', char)
    else:
        run('paragraph', run('monochrome', page))
        run('line', line)
        run('char', char)
        dt = time.perf_counter() - t0
    done = (rows_p / PAGE_HW[0] + rows_l / LINE_HW[0] + cols_c / CHAR_HW[1]) / 3.0
    return dt, done, (rows_p, rows_l, cols_c)


def _cpu_worker(job):
    os.environ['OMP_NUM_THREADS'] = '1'
    frac, train = job
    return _cpu_sample(frac, train=train)


def _sized_frac(budget_s, train):
    probe_t, _, _ = _cpu_sample(0.04, train=train)
    return float(min(1.0, max(0.04, 0.04 * budget_s / max(probe_t, 1e-3))))


def cpu_baseline(budget_s=20.0, cores=1, train=False):
    """Oracle port ("port": NumPy restatement with the reference's per-pixel loops) on a bounded
    sample: a strip of one image per sub-network, sized for ~budget_s of single-core work."""
    frac = _sized_frac(budget_s, train)
    dt, done, dims = _cpu_sample(frac, train=train)
    what = ('one Model.train step (fwd + Dice/SoftmaxCE + bwd + L2 + Adam) of each sub-network' if train
            else 'forward through Monochrome->Paragraph, Line, Char')
    return {'value': done / dt, 'unit': UNIT, 'cores': cores, 'kind': 'port',
            'sample': f'loop-form NumPy float64 port of the reference CPU path, single process, {what}: '
                      f'{dims[0]}/496 rows of one page tile, {dims[1]}/128 rows of one line tile, '
                      f'{dims[2]}/256 columns of one char line; {dt:.1f} s; images/s = mean tile fraction / time'}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    total = args.steps + args.warmup
    per_step_budget = max(2.0, min(20.0, 120.0 / max(total, 1)))
    frac = _sized_frac(per_step_budget, False)
    times, done, dims = [], None, None
    with mp.get_context('fork').Pool(cores) as pool:
        for i in range(total):
            t0 = time.perf_counter()
            res = pool.map(_cpu_worker, [(frac, False)] * cores)
            dt = time.perf_counter() - t0
            if i >= args.warmup:
                times.append(dt)
            done, dims = res[0][1], res[0][2]
        # the training step (BASELINE configs[0] / [2] on the host): one bounded sample per core
        tfrac = _sized_frac(15.0, True)
        t0 = time.perf_counter()
        tres = pool.map(_cpu_worker, [(tfrac, True)] * cores)
        twall = time.perf_counter() - t0
    sec = float(np.mean(times))
    value = cores * done / sec
    sample = (f'{cores} processes x (loop-form NumPy float64 port: {dims[0]}/496 page-tile rows through '
              f'Monochrome->Paragraph + {dims[1]}/128 line-tile rows + {dims[2]}/256 char-line columns) '
              f'per step; images/s = cores x mean tile fraction / step time')
    tdims = tres[0][2]
    train_value = cores * tres[0][1] / twall
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': sec * 1e3, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': 'BASELINE configs[1] on host cores (reference CPU algorithm, oracle port)',
                   'batch_per_gpu': args.batch},
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample},
        'cpu_baseline_train': {'value': train_value, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                               'sample': f'{cores} processes x one Model.train step (fwd + loss + bwd + L2 + Adam, '
                                         f'loop-form port) of each sub-network on {tdims[0]}/496 page-tile rows, '
                                         f'{tdims[1]}/128 line-tile rows, {tdims[2]}/256 char-line columns; '
                                         f'{twall:.1f} s wall'},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--batch', type=int, default=64, help='tiles per GPU per step')
    ap.add_argument('--math', default=os.environ.get('UOCR_MATH', 'tf32'), choices=['fp32', 'tf32'],
                    help='tf32: tcgen05 TF32 kernels for the dense contractions (default); fp32: FFMA check mode')
    ap.add_argument('--cpu-budget', type=float, default=10.0)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-train', action='store_true', help='skip the training-step measurement')
    ap.add_argument('--no-global512', action='store_true', help='skip the global-batch-512 training measurement')
    ap.add_argument('--no-fullpage', action='store_true', help='skip the full-page (configs[3]) measurement')
    ap.add_argument('--no-stages', action='store_true', help='skip the crop-stage (row f4) measurement')
    ap.add_argument('--no-gemm-peak', action='store_true', help='skip the long-GEMM TF32 rate measurement')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help="write the last timed step's predictions as DIR/<name>.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs writes the outputs of --impl b200')
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
