"""Graph executor: `Model` (a DAG of named layers, possibly nested) and `Sequential`.

Same construction and call protocol as the reference's `nn/models.py` (Model :30-484,
Sequential :487-502):

    Model(layers: dict, relations: dict, loss=...)      relations: dst -> src | [src, ...]
        int src  = model input index        int dst = model output index
        (name, i, j, ...) src = outputs i, j of a nested multi-output model
    initialize / forward / backward / compute_loss_and_gradients / train / test / predict
    params / get_weights / set_weights / nan_weights / count_parameters / regularize
    get_output_shapes / get_all_output_shapes / get_receptive_fields

Nested models are flattened to leaf layers named 'outer/inner' (these names are the keys of
model_weights.json).  Execution differs from the reference in mechanics only: instead of a
memoised recursion per call, the evaluation order is resolved once at `initialize()` and
replayed; no layer call synchronises the device, and loss values stay on the device until read.
"""
import ctypes

import numpy as np

from .._lib import ACT_LEAKY, ACT_NONE, ACT_SIGMOID, MATH_TF32, lib
from .gpu import CP, DeviceArray, LazyScalar, as_device, stream
from .help_func import make_list_if_not
from .layers import (BaseLayer, Conv2DToBatchedFixedWidthed, Convolutional2D, Flatten, FromOutput, FullyConnected,
                     LeakyRelu, Relu, Sigmoid, Upsample2D, _kmajor_copy)
from .losses import SoftmaxCrossEntropy
from .progress_tracker import track_method


class BaseModel(BaseLayer):
    def compute_loss_and_gradients(self, X, y):
        raise NotImplementedError()

    def train(self, X, y):
        loss = self.compute_loss_and_gradients(X, y)
        for param in self.params().values():
            param.update_grad()
            param.clear_grad()
        return loss

    def test(self, X, y):
        raise NotImplementedError()

    def predict(self, X):
        raise NotImplementedError()

    def params(self):
        raise NotImplementedError()

    def count_parameters(self):
        raise NotImplementedError()


def _act_code(layer):
    """(activation enum, alpha) if `layer` can run as a fused epilogue, else None."""
    if type(layer) is Sigmoid:
        return ACT_SIGMOID, 0.0
    if isinstance(layer, LeakyRelu) and layer.alpha > 0:       # Relu (alpha 0) keeps its own kernel
        return ACT_LEAKY, float(layer.alpha)
    return None


class Model(BaseModel):
    # Kernel fusion across layer boundaries (results identical up to FP32 rounding):
    #   training + inference : Convolutional2D -> LeakyRelu as one kernel (the activation's
    #                          backward is then evaluated from its OUTPUT, exact for alpha > 0)
    #   inference only       : Convolutional2D -> Sigmoid as one kernel
    #   inference only       : Upsample2D(2) -> Convolutional2D folded into the conv's addressing;
    #                          3x3 conv (1->C) -> act -> 3x3 conv (C->1) [-> act] as one kernel with
    #                          the C-channel map kept in registers (Monochrome)
    # Fused-away tensors are absent (None) from `layers_outputs`; set `fusion = False` (class or
    # instance) before initialize() to get every per-layer output like the reference.
    fusion = True
    # Optional whole-network inference kernel: a callable (model, inputs) -> list of outputs or None
    # (None = geometry not supported, run the layer plan).  Set by builders that know the topology
    # (my_model._make_hourglass -> HourglassFusion); only consulted when `fusion` is on and training
    # is off, so training, gradient checks and `fusion = False` see the plain layer graph.
    infer_fusion = None
    # False: skip the gradient w.r.t. the model INPUTS (the reference always computes it,
    # models.py:207-230, but a training step never uses it); `input_grads` entries are then None
    compute_input_grads = True

    def __init__(self, layers, relations, loss=SoftmaxCrossEntropy(), *args, **kwargs):
        super().__init__(*args, **kwargs)
        if not isinstance(layers, dict):
            raise TypeError(f'layers argument must be dict, found: {type(layers).__name__}')
        if not isinstance(relations, dict):
            raise TypeError(f'relations argument must be dict, found: {type(relations).__name__}')
        self.ravelled_layers = layers
        self.ravelled_relations = relations
        self.layers = None
        self.relations = None
        self.relations_backward = {}
        self.inputs_count = max(v for v in relations.values() if isinstance(v, int)) + 1
        self.outputs_count = max(k for k in relations if isinstance(k, int)) + 1
        self.layers_outputs = {}
        self.loss = loss
        self.input_grads = {}
        self.is_initialized = False
        self._receptive_fields = {}
        self._order = None
        self.unravel_model()

    # ---- structure ----------------------------------------------------------------
    def unravel_model(self):
        """Flattens nested Models: their leaf layers become 'name/leaf', their int inputs are
        wired to this model's sources and their int outputs replace `name` / `(name, i, ...)`
        wherever it is consumed (reference :109-158)."""
        relations = {dst: list(make_list_if_not(src)) for dst, src in self.ravelled_relations.items()}
        leaves = {}
        for name, layer in self.ravelled_layers.items():
            if not isinstance(layer, Model):
                leaves[name] = layer
                continue
            layer.unravel_model()
            for leaf_name, leaf in layer.layers.items():
                leaves[f'{name}/{leaf_name}'] = leaf
            feeds = relations[name]
            outputs = {}
            for dst, srcs in layer.relations.items():
                wired = [feeds[s] if isinstance(s, int) else f'{name}/{s}' for s in srcs]
                if isinstance(dst, int):
                    outputs[dst] = wired
                else:
                    relations[f'{name}/{dst}'] = wired
            del relations[name]
            for dst, srcs in relations.items():
                rewired = []
                for src in srcs:
                    if isinstance(src, str) and src == name:
                        for out_id in range(layer.get_outputs_count()):
                            rewired.extend(outputs[out_id])
                    elif isinstance(src, tuple) and len(src) > 1 and src[0] == name:
                        for out_id in src[1:]:
                            rewired.extend(outputs[out_id])
                    else:
                        rewired.append(src)
                relations[dst] = rewired
        if self.layers is None:
            self.layers = leaves
        self.relations = relations
        for name, layer in self.layers.items():
            layer._set_name(name)

    def get_leaf_layers(self):
        return self.layers

    def __getitem__(self, key):
        return self.layers[key]

    def _output_keys(self):
        return sorted(k for k in self.relations if isinstance(k, int))

    def _resolve_order(self):
        """Depth-first from the outputs: evaluation order of the layers that feed an output."""
        order, state = [], {}

        def visit(name):
            if isinstance(name, int) and name not in self.relations:
                return
            if state.get(name) == 'done':
                return
            if state.get(name) == 'open':
                raise RecursionError(f'Looped on {name} layer, check relations')
            state[name] = 'open'
            for src in self.relations[name]:
                if not isinstance(src, int):
                    visit(src)
            state[name] = 'done'
            if not isinstance(name, int):
                order.append(name)

        for key in self._output_keys():
            state.pop(key, None)
            for src in self.relations[key]:
                if not isinstance(src, int):
                    visit(src)
        return order

    def initialize(self, input_shapes):
        input_shapes = make_list_if_not(input_shapes)
        self.input_shapes = input_shapes
        self._order = self._resolve_order()
        self.relations_backward = {}
        shapes = {}

        def shape_of(src):
            if isinstance(src, int):
                return input_shapes[src]
            s = shapes[src]
            return s[0] if isinstance(s, list) else s

        for name in self._order + self._output_keys():
            srcs = self.relations[name]
            for i, src in enumerate(srcs):
                self.relations_backward.setdefault(src, {})[name] = i
            if isinstance(name, int):
                continue
            in_shapes = [shape_of(src) for src in srcs]
            layer = self.layers[name]
            if not layer.is_initialized:
                layer.initialize(in_shapes)
            shapes[name] = layer.get_output_shapes(in_shapes)

        never = [n for n in self.layers if n not in shapes]
        if never:
            print(f'These layers have never been visited: {never}')
        self._plan_train = self._make_plan(training=True)
        self._plan_infer = self._make_plan(training=False)
        if self.fusion and self.infer_fusion is None:
            # whole-network inference kernels are recognised from the topology, so networks built by the reference's
            # own my_model/model.py (which knows nothing about them) get them as well
            self.infer_fusion = HourglassFusion.detect(self)
        self._fusion_planned = bool(self.fusion)                    # like the plans: fixed at initialize
        self.is_initialized = True

    # ---- fusion planning ----------------------------------------------------------
    def _sole_consumer(self, name):
        """The single layer consuming `name`'s output (as its only input), else None."""
        users = self.relations_backward.get(name, {})
        if len(users) != 1:
            return None
        (dst, _), = users.items()
        if isinstance(dst, int) or len(self.relations[dst]) != 1 or dst not in self.layers:
            return None
        return dst

    def _make_plan(self, training, ragged=False):
        """`ragged`: the inference plan of `predict_ragged`, without the Monochrome pair kernel, whose C-channel
        intermediate stays on chip where it cannot be zeroed outside each image's extent."""
        plan, taken = [], set()
        for name in self._order:
            if name in taken:
                continue
            layer = self.layers[name]
            step = None
            if self.fusion and len(self.relations[name]) == 1:
                ups = None
                conv_name = name
                if type(layer) is Upsample2D and layer.scale_factor == (2, 2):
                    nxt = self._sole_consumer(name)
                    # training: only where the conv's weight gradient can read through the upsampling
                    if (nxt is not None and type(self.layers[nxt]) is Convolutional2D
                            and (not training or self.layers[nxt].supports_upsampled_input_grad())):
                        ups, conv_name = name, nxt
                conv = self.layers[conv_name]
                if type(conv) is Convolutional2D or (type(conv) is FullyConnected and ups is None):
                    act_name = self._sole_consumer(conv_name)
                    act = _act_code(self.layers[act_name]) if act_name is not None else None
                    # training: a fused Sigmoid would have to be differentiated from its output
                    # y * (1 - y), which flushes saturated gradients (|x| > 17) to zero in FP32
                    # while the reference's exp(-x) / (1 + exp(-x))^2 keeps them; LeakyRelu's
                    # derivative from the output is exact (sign(y) == sign(x))
                    if act is None or (training and act[0] != ACT_LEAKY):
                        act_name = None
                    pair = None
                    if (ups is None and act_name is not None and type(conv) is Convolutional2D and not ragged
                            and self._pair_head(conv)
                            and (not training or act[0] == ACT_LEAKY)):
                        c2_name = self._sole_consumer(act_name)
                        if c2_name is not None and self._pair_tail(conv, self.layers[c2_name]):
                            a2_name = self._sole_consumer(c2_name) if not training else None
                            a2 = _act_code(self.layers[a2_name]) if a2_name is not None else None
                            pair = (c2_name, a2_name if a2 is not None else None)
                    chain = None
                    if (not training and type(conv) is FullyConnected and act_name is not None
                            and conv.n_output == self.FC_CHAIN_HIDDEN):
                        # inference: FullyConnected(-> 128) + activation + FullyConnected as one kernel whose hidden
                        # tile stays in shared memory (uocr_fc_chain2_fwd): Char dense_2 + leaky_relu_2 + dense_3
                        nxt = self._sole_consumer(act_name)
                        if nxt is not None and type(self.layers[nxt]) is FullyConnected:
                            after = self._sole_consumer(nxt)
                            if after is None or _act_code(self.layers[after]) is None:
                                chain = nxt
                    if pair is not None:
                        step = ('pair', conv_name, act_name, pair[0], pair[1])
                    elif chain is not None:
                        step = ('fcchain', conv_name, act_name, chain)
                    elif ups is not None or act_name is not None:
                        step = ('conv', ups, conv_name, act_name)
            if (step is None and self.fusion and not training and type(layer) is Conv2DToBatchedFixedWidthed
                    and len(self.relations[name]) == 1):
                # inference: window batching + Flatten + FullyConnected (+ activation) as one GEMM whose A operand
                # is gathered from the un-windowed tensor (uocr_window_fc_fwd)
                flat = self._sole_consumer(name)
                fc = self._sole_consumer(flat) if flat is not None and type(self.layers[flat]) is Flatten else None
                if fc is not None and type(self.layers[fc]) is FullyConnected:
                    act_name = self._sole_consumer(fc)
                    if act_name is not None and _act_code(self.layers[act_name]) is None:
                        act_name = None
                    step = ('winfc', name, flat, fc, act_name)
            if step is None:
                step = ('layer', name)
            plan.append(step)
            taken.update(n for n in step[1:] if n is not None)
        return plan

    @staticmethod
    def _pair_head(conv):
        return (conv.kernel_size == (3, 3) and conv.padding == (1, 1) and conv.stride == (1, 1)
                and conv.in_channels == 1 and conv.padding_value == 0 and conv.bias
                and conv.out_channels <= 256)

    @staticmethod
    def _pair_tail(head, conv):
        return (type(conv) is Convolutional2D and conv.kernel_size == (3, 3)
                and conv.padding == (1, 1) and conv.stride == (1, 1) and conv.out_channels == 1
                and conv.in_channels == head.out_channels and conv.padding_value == 0 and conv.bias)

    # ---- execution ----------------------------------------------------------------
    @track_method('forward')
    def forward(self, inputs, training=True, clear_grads=True):
        """`clear_grads=False` skips the reference's per-layer `clear_grads()` before each layer's
        forward (models.py:188) -- for callers that zero one flat gradient buffer themselves."""
        inputs = make_list_if_not(inputs)
        if not self.is_initialized:
            self.initialize_from_X(inputs)
        if not training and self._fusion_planned and self.infer_fusion is not None:
            fused = self.infer_fusion(self, inputs)
            if fused is not None:
                self.layers_outputs = {**{name: None for name in self.layers},
                                       **{k: fused[k] for k in range(self.outputs_count)}}
                return fused

        outputs = self._run_steps(self._plan_train if training else self._plan_infer, inputs, training, clear_grads)
        self.layers_outputs = outputs
        return [outputs[k] for k in range(self.outputs_count)]

    def _run_steps(self, plan, inputs, training, clear_grads, after_step=None):
        """Runs `plan` on `inputs` -> {layer name / output index: value}; `after_step(step, outputs)` after each step."""
        outputs = {}

        def value_of(src):
            return inputs[src] if isinstance(src, int) else outputs[src]

        for step in plan:
            kind = step[0]
            if kind == 'layer':
                name = step[1]
                layer = self.layers[name]
                if clear_grads:
                    layer.clear_grads()                            # reference :188
                out = layer.forward([value_of(src) for src in self.relations[name]])
                outputs[name] = out[0] if isinstance(out, list) else out
            elif kind == 'conv':
                self._run_fused_conv(step, value_of, outputs, training, clear_grads)
            elif kind == 'winfc':
                self._run_winfc(step, value_of, outputs)
            elif kind == 'fcchain':
                self._run_fcchain(step, value_of, outputs)
            else:
                if clear_grads:                                    # reference :188, for every member of the fused pair
                    for member in step[1:]:
                        if member is not None:
                            self.layers[member].clear_grads()
                self._run_pair(step, value_of, outputs, training)
            if after_step is not None:
                after_step(step, outputs)
        for key in self._output_keys():
            outputs[key] = value_of(self.relations[key][0])
        return outputs

    def _run_fused_conv(self, step, value_of, outputs, training, clear_grads=True):
        _, ups_name, conv_name, act_name = step
        first = ups_name if ups_name is not None else conv_name
        X = as_device(value_of(self.relations[first][0]))
        conv = self.layers[conv_name]
        act_layer = self.layers[act_name] if act_name is not None else None
        act, alpha = _act_code(act_layer) if act_layer is not None else (ACT_NONE, 0.0)
        tracked = [self.layers[n] for n in (ups_name, conv_name, act_name) if n is not None]
        if clear_grads:
            for layer in tracked:
                layer.clear_grads()
        last = tracked[-1]
        if training and ups_name is not None:
            if X.shape[2] % 2:                   # the upsampled-input wgrad kernel needs Wo % 4 == 0
                X = as_device(self.layers[ups_name].forward([X])[0])
                outputs[ups_name], ups_name = X, None
            else:
                self.layers[ups_name]._mem[0] = X.shape         # all Upsample2D._backward needs
        last.progress_tracker.start_tracking(last.name, 'forward')
        y = conv._forward(X, 0, act=act, alpha=alpha, in_upsample=2 if ups_name is not None else 1,
                          save=training)
        last.progress_tracker.stop_tracking(last.name, 'forward')
        if training and act_layer is not None:
            act_layer._mem[0] = FromOutput(y)
        for n in (ups_name, conv_name, act_name):
            if n is not None:
                outputs[n] = None
        outputs[act_name if act_name is not None else conv_name] = y

    def _run_winfc(self, step, value_of, outputs):
        """Inference only: Conv2DToBatchedFixedWidthed -> Flatten -> FullyConnected (-> activation)."""
        _, win_name, flat_name, fc_name, act_name = step
        X = as_device(value_of(self.relations[win_name][0]))
        win, fc = self.layers[win_name], self.layers[fc_name]
        n, h, w, c = X.shape
        names = [nm for nm in (win_name, flat_name, fc_name, act_name) if nm is not None]
        if h != 1 or win.width * c != fc.n_input:          # not the Char head's geometry: layer by layer
            cur = X
            for nm in names:
                out = self.layers[nm].forward([cur])
                cur = out[0] if isinstance(out, list) else out
                outputs[nm] = cur
            return
        assert w >= win.width, f'Input width must be >= than output width, found: {w} < {win.width}'
        act, alpha = _act_code(self.layers[act_name]) if act_name is not None else (ACT_NONE, 0.0)
        last = self.layers[names[-1]]
        last.progress_tracker.start_tracking(last.name, 'forward')
        y = DeviceArray((n * w, fc.n_output))
        wt = _kmajor_copy(fc, fc.w.value, fc.n_input, fc.n_output) if CP.math_mode == MATH_TF32 else None
        lib.uocr_window_fc_fwd(X.ptr, fc.w.value.ptr, wt.ptr if wt is not None else None, y.ptr, n, w, c, win.width,
                               fc.n_output, act, float(alpha), CP.math_mode, stream())
        last.progress_tracker.stop_tracking(last.name, 'forward')
        for nm in names:
            outputs[nm] = None
        outputs[names[-1]] = y

    FC_CHAIN_HIDDEN = 128                                # hidden width the two-layer kernel is built for

    def _run_fcchain(self, step, value_of, outputs):
        """Inference only: FullyConnected -> activation -> FullyConnected (uocr_fc_chain2_fwd; any geometry or math mode
        the one-kernel path does not cover runs as two GEMMs inside the library)."""
        _, fc1_name, act_name, fc2_name = step
        X = as_device(value_of(self.relations[fc1_name][0]))
        fc1, fc2 = self.layers[fc1_name], self.layers[fc2_name]
        assert len(X.shape) == 2 and X.shape[1] == fc1.n_input, f'{fc1_name}: expected (batch, {fc1.n_input}), got {X.shape}'
        act, alpha = _act_code(self.layers[act_name])
        fc2.progress_tracker.start_tracking(fc2.name, 'forward')
        y = DeviceArray((X.shape[0], fc2.n_output))
        tf32 = CP.math_mode == MATH_TF32
        w1t = _kmajor_copy(fc1, fc1.w.value, fc1.n_input, fc1.n_output) if tf32 else None
        w2t = _kmajor_copy(fc2, fc2.w.value, fc2.n_input, fc2.n_output) if tf32 else None
        lib.uocr_fc_chain2_fwd(X.ptr, fc1.w.value.ptr, w1t.ptr if w1t is not None else None, fc2.w.value.ptr,
                               w2t.ptr if w2t is not None else None, y.ptr, X.shape[0], fc1.n_input, fc1.n_output,
                               fc2.n_output, act, float(alpha), CP.math_mode, stream())
        fc2.progress_tracker.stop_tracking(fc2.name, 'forward')
        outputs[fc1_name] = outputs[act_name] = None
        outputs[fc2_name] = y

    def _run_pair(self, step, value_of, outputs, training=False):
        _, c1_name, a1_name, c2_name, a2_name = step
        X = as_device(value_of(self.relations[c1_name][0]))
        c1, c2 = self.layers[c1_name], self.layers[c2_name]
        if training:
            c1._mem[0] = X                                      # all the fused backward needs
        act1, alpha1 = _act_code(self.layers[a1_name])
        act2, alpha2 = _act_code(self.layers[a2_name]) if a2_name is not None else (ACT_NONE, 0.0)
        n, h, w, cin = X.shape
        assert cin == 1, f'input has {cin} channels, layer expects 1'
        last = self.layers[a2_name if a2_name is not None else c2_name]
        last.progress_tracker.start_tracking(last.name, 'forward')
        y = DeviceArray((n, h, w, 1))
        lib.uocr_conv3x3_pair_fwd(X.ptr, c1.w.value.ptr, c1.b.value.ptr, c2.w.value.ptr, c2.b.value.ptr,
                                  y.ptr, n, h, w, c1.out_channels, act1, alpha1, act2, alpha2, CP.math_mode,
                                  stream())
        last.progress_tracker.stop_tracking(last.name, 'forward')
        for nme in (c1_name, a1_name, c2_name, a2_name):
            if nme is not None:
                outputs[nme] = None
        outputs[a2_name if a2_name is not None else c2_name] = y

    @track_method('backward')
    def backward(self, grads, on_layer_done=None):
        """`on_layer_done(name)` is called as soon as the parameter gradients of layer `name` are final (its backward
        kernels are queued on the current stream) -- the data-parallel step starts that layer's gradient allreduce
        there, while the rest of backward runs."""
        grads = make_list_if_not(grads)
        produced = {}                                               # layer -> list of input grads
        done = on_layer_done if on_layer_done is not None else (lambda name: None)

        def incoming(name):
            parts = []
            for dst, slot in self.relations_backward[name].items():
                parts.append(grads[dst] if isinstance(dst, int) else produced[dst][slot])
            return sum(parts)                                       # 0 + g1 (+ g2 ...), reference :218

        pairs = {}                                                  # member layer -> ('pair', c1, a1, c2, None)
        for step in self._plan_train:
            if step[0] == 'pair':
                for member in step[1:4]:
                    pairs[member] = step
        stash = {}
        for name in reversed(self._order):
            step = pairs.get(name)
            layer = self.layers[name]
            if step is None:
                first = all(isinstance(src, int) for src in self.relations[name])
                if first and not self.compute_input_grads and hasattr(layer, 'backward_params_only'):
                    layer.backward_params_only(incoming(name))
                    produced[name] = [None] * len(self.relations[name])
                else:
                    produced[name] = make_list_if_not(layer.backward(incoming(name)))
                done(name)
            elif name == step[3]:                                   # conv_2: keep its output gradient
                stash[step[1]] = incoming(name)
                produced[name] = [None]
            elif name == step[2]:                                   # the activation in between
                produced[name] = [None]
            else:                                                   # conv_1: the fused backward
                first = all(isinstance(src, int) for src in self.relations[name])
                produced[name] = [self._pair_backward(step, stash.pop(name),
                                                      need_dx=self.compute_input_grads or not first)]
                done(step[3])
                done(name)
        for key in range(self.inputs_count):
            self.input_grads[key] = incoming(key) if self.compute_input_grads else None
        return [self.input_grads[k] for k in range(self.inputs_count)]

    def _pair_backward(self, step, grad, need_dx=True):
        _, c1_name, a1_name, c2_name, _ = step
        c1, c2 = self.layers[c1_name], self.layers[c2_name]
        act1, alpha1 = _act_code(self.layers[a1_name])
        X = c1._mem.pop(0)
        grad = as_device(grad)
        n, h, w, _ = X.shape
        need = ctypes.c_size_t(0)
        lib.uocr_conv3x3_pair_bwd_workspace(n, h, w, c1.out_channels, ctypes.byref(need))
        ws = DeviceArray(((need.value + 3) // 4,))
        dx = DeviceArray(X.shape) if need_dx else None
        tracker = c1.progress_tracker
        tracker.start_tracking(c1.name, 'backward')
        lib.uocr_conv3x3_pair_bwd_mode(X.ptr, c1.w.value.ptr, c1.b.value.ptr, c2.w.value.ptr, grad.ptr,
                                       dx.ptr if need_dx else None, c1.w.grad.ptr, c1.b.grad.ptr, c2.w.grad.ptr,
                                       c2.b.grad.ptr, n, h, w, c1.out_channels, act1, alpha1, 1, ws.ptr, need.value,
                                       CP.math_mode, stream())
        tracker.stop_tracking(c1.name, 'backward')
        return dx

    def _loss_for(self, key):
        return self.loss[key] if isinstance(self.loss, list) else self.loss

    def compute_loss_and_gradients(self, X, y):
        X, y = make_list_if_not(X), make_list_if_not(y)
        if self._flat:
            self._flat.clean = False                                # gradients are about to be left in param.grad
        predicted = self.forward(X)
        losses, gradients = [], []
        for key in range(self.outputs_count):
            loss, grad = self._loss_for(key)(predicted[key], y[key])
            losses.append(loss)
            gradients.append(grad)
        self.backward(gradients)
        return {'output_losses': losses, 'regularization_loss': self.regularize()}

    # `Model.train` (reference :250-254) = compute_loss_and_gradients -> update_grads -> clear_grads: per parameter
    # tensor one regulariser kernel, one Adam kernel and one memset (the reference: ~12 CuPy kernels and a host sync
    # each).  When the model is what my_model builds -- one shared Adam, L2 or no regulariser, everything trainable
    # (`FlatParameters.eligible`) -- the same step runs on flat buffers: forward + loss + backward, then ONE fused
    # L2 + Adam launch per regularisation group and ONE memset.  Same numbers (tests/test_gpu_parity.py); set
    # `fused_update = False` (class or instance) for the per-parameter route.
    fused_update = True
    _flat = None

    def fused_optimizer(self):
        """The shared Adam instance if this model qualifies for the fused update right now, else None."""
        from .flat import FlatParameters
        if not self.is_initialized:
            return None
        return FlatParameters.eligible(self)

    def flat_parameters(self):
        """The model's `FlatParameters` (created on first use), or None if it does not qualify."""
        if self._flat is None:
            from .flat import FlatParameters
            if self.fused_optimizer() is None:
                return None
            self._flat = FlatParameters(self)
        return self._flat

    def train_fused(self, X, y, reduce_gradients=None, grad_scale=1.0, on_layer_done=None):
        """One training step on the flat buffers.  `reduce_gradients()` runs between backward and the update (the
        data-parallel allreduce); returns the same dict as `train`."""
        opt, flat = self.fused_optimizer(), self.flat_parameters()
        assert flat is not None and opt is not None, 'model does not qualify for the fused update'
        if not flat.attached():
            flat.adopt()
        if not flat.clean:
            flat.zero_grads()
        X, y = make_list_if_not(X), make_list_if_not(y)
        keep, self.compute_input_grads = self.compute_input_grads, False    # `train` never surfaces dL/dX (:250-254)
        try:
            predicted = self.forward(X, clear_grads=False)
            losses, gradients = [], []
            for key in range(self.outputs_count):
                loss, grad = self._loss_for(key)(predicted[key], y[key])
                losses.append(loss)
                gradients.append(grad)
            flat.clean = False
            self.backward(gradients, on_layer_done=on_layer_done)
        finally:
            self.compute_input_grads = keep
        if reduce_gradients is not None:
            reduce_gradients()
        reg = flat.update(opt, grad_scale)
        self.input_grads = {}
        return {'output_losses': losses, 'regularization_loss': reg}

    def train(self, X, y):
        if self.fused_update and self.fused_optimizer() is not None:
            return self.train_fused(X, y)
        losses = self.compute_loss_and_gradients(X, y)
        self.update_grads()
        self.clear_grads()
        return losses

    def test(self, X, y):
        X, y = make_list_if_not(X), make_list_if_not(y)
        predicted = self.forward(X, training=False)
        losses = []
        for key in range(self.outputs_count):
            fn = self._loss_for(key)
            try:
                loss, _ = fn(predicted[key], y[key], want_grad=False)
            except TypeError:                                       # user-supplied loss object
                loss, _ = fn(predicted[key], y[key])
            losses.append(loss)
        return {'output_losses': losses}

    def predict(self, X):
        return self.forward(X, training=False)

    # ---- ragged batches -----------------------------------------------------------
    # Layers whose zero padding makes a canvas of zero-padded images exact (DESIGN.md §3).  Relu is listed apart from
    # LeakyRelu because the check is by exact type.
    RAGGED_LAYERS = (Convolutional2D, Upsample2D, LeakyRelu, Relu, Sigmoid, Conv2DToBatchedFixedWidthed, Flatten,
                     FullyConnected)
    _plan_ragged = None

    def ragged_analysis(self, canvas_shape, extents):
        """Host-side analysis of a ragged batch: a canvas (N, H, W, C) holding image i in [i, :h_i, :w_i, :] with
        (h_i, w_i) = extents[i].  Raises ValueError for extents outside the canvas and for layers a ragged batch cannot
        run through.  -> (extents as int64 (N, 2), {layer name: ('hw', (N, 2) per-image (h, w) of its output, the canvas
        output's (H, W)) or ('rows', (N, 2) [first, end) row range of each image, None)}).  The per-image shapes are the model's own shape analysis
        of (1, h_i, w_i, C), one analysis per distinct extent.  After a Conv2DToBatchedFixedWidthed the batch axis holds
        one row per window: image i owns rows [i * W, i * W + w_i) of it, W and w_i the canvas and image widths there."""
        assert self.is_initialized, 'The model must be initialized before calling this method'
        for name, layer in self.layers.items():
            if type(layer) not in self.RAGGED_LAYERS:
                raise ValueError(f'{name}: {type(layer).__name__} is not supported on ragged batches')
            if type(layer) is Convolutional2D and layer.padding_value != 0:
                raise ValueError(f'{name}: padding_value {layer.padding_value} != 0 is not supported on ragged batches')
        if self.inputs_count != 1:
            raise ValueError(f'ragged batches need a model with one input, this one has {self.inputs_count}')
        shape = tuple(int(v) for v in canvas_shape)
        if len(shape) != 4:
            raise ValueError(f'a ragged canvas is (N, H, W, C), got shape {shape}')
        n, H, W, C = shape
        ext = np.asarray(extents)
        if ext.shape != (n, 2) or not (ext.dtype.kind in 'iu' or ext.size == 0):
            raise ValueError(f'extents must be an integer ({n}, 2) array, got {ext.dtype} {ext.shape}')
        ext = ext.astype(np.int64)
        bad = np.flatnonzero((ext[:, 0] < 1) | (ext[:, 0] > H) | (ext[:, 1] < 1) | (ext[:, 1] > W))
        if bad.size:
            i = int(bad[0])
            raise ValueError(f'extent {i} = {tuple(int(v) for v in ext[i])} is outside the {H} x {W} canvas')
        canvas_shapes = self.get_all_output_shapes([shape])[1]
        per_extent = {}
        for h, w in sorted(set(map(tuple, ext.tolist()))):
            try:
                per_extent[h, w] = self.get_all_output_shapes([(1, h, w, C)])[1]
            except AssertionError as e:
                raise ValueError(f'extent {h} x {w}: {e}') from None
        keys = [tuple(e) for e in ext.tolist()]
        modes = {}

        def mode_of(src):
            return ('hw', ext, (H, W)) if isinstance(src, int) else modes[src]

        def canvas_of(src):
            return shape if isinstance(src, int) else canvas_shapes[src][0]

        for name in self._order:
            layer, srcs = self.layers[name], self.relations[name]
            kinds = {mode_of(src)[0] for src in srcs}
            if kinds == {'rows'}:
                modes[name] = mode_of(srcs[0])
            elif kinds != {'hw'}:
                raise ValueError(f'{name}: mixes image maps and window rows')
            elif type(layer) is Conv2DToBatchedFixedWidthed:
                (_, hc, wc, _), table = canvas_of(srcs[0]), mode_of(srcs[0])[1]
                if (table[:, 0] != hc).any():
                    raise ValueError(f'{name}: windows of images shorter than the canvas would carry its padding')
                first = np.arange(n, dtype=np.int64) * wc
                modes[name] = ('rows', np.stack([first, first + table[:, 1]], axis=1), None)
            elif type(layer) in (Flatten, FullyConnected):
                raise ValueError(f'{name}: {type(layer).__name__} of a ragged image map would mix in its padding')
            else:
                table = np.array([per_extent[k][name][0][1:3] for k in keys], dtype=np.int64).reshape(n, 2)
                _, hc, wc, _ = canvas_of(name)
                if (table[:, 0] > hc).any() or (table[:, 1] > wc).any():
                    raise ValueError(f'{name}: an image output is larger than the canvas output {hc} x {wc}')
                modes[name] = ('hw', table, (hc, wc))
        return ext, modes

    def predict_ragged(self, canvas, extents):
        """Inference on a ragged batch: `canvas` (N, H, W, C) device (or host) array, zero outside each image, image i
        in canvas[i, :h_i, :w_i, :]; `extents` host (N, 2) integers (h_i, w_i).  -> (outputs, output extents): one output
        canvas per model output and, per output, an (N, 2) int64 array -- (h_i, w_i) of image i's region for an image
        map, [first, end) of image i's rows after a Conv2DToBatchedFixedWidthed (see `ragged_analysis`).  Image i's
        region equals `predict` on that image alone, up to the rounding of shape-dependent kernel choices, and image maps
        are 0 outside it.  Every step that outputs an image map is followed by uocr_zero_outside_hw_f32 where some extent
        is smaller than the canvas; fused steps that keep a spatial map on chip step aside for their materialising
        equivalents (the Paragraph one-kernel, the Monochrome pair kernel), the Line one-kernel runs its ragged variant
        when every extent is a multiple of 4.  Extents and layers are checked before anything is launched."""
        ext, modes = self.ragged_analysis(canvas.shape, extents)
        out_names = [self.relations[k][0] for k in range(self.outputs_count)]

        def out_table(src):
            return ext.copy() if isinstance(src, int) else modes[src][1].copy()

        # every extent table a kernel reads, uploaded in one copy: the input's, then one per masked output
        tables, offsets = [ext], {}
        for name in self._order:
            kind, table, canvas_hw = modes[name]
            if kind == 'hw' and ((table[:, 0] < canvas_hw[0]) | (table[:, 1] < canvas_hw[1])).any():
                offsets[name] = sum(t.size for t in tables)
                tables.append(table)
        dev = DeviceArray.from_host(np.concatenate(tables).astype(np.int32), np.int32)
        X = as_device(canvas)
        if self._fusion_planned and isinstance(self.infer_fusion, HourglassFusion):
            fused = self.infer_fusion(self, [X], ext, dev.ptr)
            if fused is not None:
                self.layers_outputs = {**{name: None for name in self.layers}, 0: fused[0]}
                return fused, [out_table(out_names[0])]
        if self._plan_ragged is None:
            self._plan_ragged = self._make_plan(training=False, ragged=True) if self._fusion_planned else self._plan_infer

        def mask(step, outputs):
            name = [m for m in step[1:] if m is not None][-1]
            if name in offsets:
                y = outputs[name]
                lib.uocr_zero_outside_hw_f32(y.ptr, dev.ptr + 4 * offsets[name], *y.shape, stream())

        outputs = self._run_steps(self._plan_ragged, [X], False, True, after_step=mask)
        self.layers_outputs = outputs
        return [outputs[k] for k in range(self.outputs_count)], [out_table(src) for src in out_names]

    def update_grads(self):
        if not self.trainable:
            return
        for layer in self.layers.values():
            layer.update_grads()

    def clear_grads(self):
        for layer in self.layers.values():
            layer.clear_grads()
        self.input_grads = {}

    def regularize(self, loss_dev=None):
        regularised = [l for l in self.layers.values() if getattr(l, 'regularizer', None) is not None]
        if not regularised:
            return 0
        own = loss_dev is None
        if own:
            loss_dev = DeviceArray.zeros((1,))
        for layer in regularised:
            layer.regularize(loss_dev)
        return LazyScalar(loss_dev) if own else 0

    # ---- parameters ---------------------------------------------------------------
    def params(self):
        return {f'{layer_name}/{name}': param
                for layer_name, layer in self.layers.items()
                for name, param in layer.params().items()}

    def get_weights(self):
        weights = {name: layer.get_weights() for name, layer in self.layers.items()}
        return {name: w for name, w in weights.items() if w != {}}

    def set_weights(self, weights):
        for name, layer in self.layers.items():
            layer_weights = weights.get(name, None)
            if layer_weights is not None:
                layer.set_weights(layer_weights)

    def nan_weights(self):
        return any(layer.nan_weights() for layer in self.layers.values())

    def count_parameters(self):
        return sum(layer.count_parameters() for layer in self.layers.values())

    def init_progress_tracker(self, progress_tracker, model_name='model'):
        if self.name is None:
            self.name = model_name
        self.progress_tracker = progress_tracker
        self.progress_tracker.register_layer(self.name)
        for layer in self.layers.values():
            layer.init_progress_tracker(progress_tracker, None)

    # ---- shape analysis -----------------------------------------------------------
    def get_all_output_shapes(self, input_shapes):
        input_shapes = make_list_if_not(input_shapes)

        def plain(shapes):
            out = []
            for shape in make_list_if_not(shapes):
                assert isinstance(shape, tuple)
                out.append(tuple(int(x) for x in shape))
            return out

        per_layer, extra = {}, {}

        def shape_of(src):
            if isinstance(src, int):
                return input_shapes[src]
            s = per_layer[src]
            return s[0] if isinstance(s, list) else s

        order = self._order if self._order is not None else self._resolve_order()
        for name in order:
            ins = [shape_of(src) for src in self.relations[name]]
            own, nested = self.layers[name].get_all_output_shapes(ins)
            per_layer[name] = plain(own)
            extra.update({f'{name}/{k}': plain(v) for k, v in nested.items()})
        result = [shape_of(self.relations[key][0]) for key in range(self.outputs_count)]
        extra.update(per_layer)
        return plain(result), extra

    def get_output_shapes(self, input_shapes):
        return self.get_all_output_shapes(input_shapes)[0]

    def get_outputs_count(self):
        return self.outputs_count

    def is_fully_convolutional(self):
        return all(layer.is_fully_convolutional() for layer in self.layers.values())

    def changes_receptive_field(self):
        return any(layer.changes_receptive_field() for layer in self.layers.values())

    # ---- receptive fields (reference :340-432) ------------------------------------
    def _rf_relations(self):
        """Relations with every layer that does not change the receptive field spliced out."""
        if 'relations' in self._receptive_fields:
            return self._receptive_fields['relations']
        rel = {dst: list(srcs) for dst, srcs in self.relations.items()}
        for name, layer in self.layers.items():
            if layer.changes_receptive_field() or name not in rel:
                continue
            sources = rel.pop(name)
            for dst in rel:
                spliced = []
                for src in rel[dst]:
                    spliced.extend(sources if src == name else [src])
                rel[dst] = spliced
        self._receptive_fields['relations'] = rel
        return rel

    def _get_receptive_field(self, axis, position, output_id):
        key = (axis, position, output_id)
        if key in self._receptive_fields:
            return self._receptive_fields[key]
        rel = self._rf_relations()
        memo = {}

        def points(name, pos):
            if (name, pos) in memo:
                return memo[name, pos]
            own = {0: {pos}} if isinstance(name, int) else self.layers[name]._get_receptive_field(axis, pos, 0)
            acc = {k: set() for k in range(self.inputs_count)}
            for slot, src in enumerate(rel[name]):
                if isinstance(src, int):
                    acc[src].update(own[slot])
                    continue
                for p in own[slot]:
                    for in_key, pts in points(src, p).items():
                        acc[in_key].update(pts)
            memo[name, pos] = acc
            return acc

        for name in rel:
            self._receptive_fields[name, axis] = points(name, 0)
        return points(rel[output_id][0], position)

    def get_receptive_fields(self):
        assert self.is_initialized, 'The model must be initialized before calling this method'
        assert self.is_fully_convolutional(), (
            'This method is only available for Fully Convolutional Networks (FCN)')
        for output_id in range(self.get_outputs_count()):
            for axis in range(2):
                self._get_receptive_field(axis, 0, output_id)
        result = {}
        for name in self._receptive_fields['relations']:
            if isinstance(name, int):
                continue
            rf_y, rf_x = self._receptive_fields[name, 0], self._receptive_fields[name, 1]
            result[name] = {}
            for in_id in rf_y:
                ys, xs = rf_y[in_id], rf_x[in_id]
                if not ys or not xs:
                    continue
                result[name][f'input {in_id}'] = {
                    'cnt': (len(ys), len(xs)),
                    'y': (min(ys), max(ys)),
                    'x': (min(xs), max(xs)),
                    'is_solid_y': len(ys) == max(ys) - min(ys) + 1,
                    'is_solid_x': len(xs) == max(xs) - min(xs) + 1,
                }
        self._clear_receptive_fields_info()
        return result

    def _clear_receptive_fields_info(self):
        for layer in self.layers.values():
            layer._clear_receptive_fields_info()
        self._receptive_fields = {}


class Sequential(Model):
    """Chain of layers named '{i}_{ClassName}' (reference :487-502)."""

    def __init__(self, layers, *args, **kwargs):
        if not isinstance(layers, list):
            raise TypeError(f'layers argument must be list, found: {type(layers).__name__}')
        named, relations, prev = {}, {}, 0
        for i, layer in enumerate(layers):
            name = f'{i}_{type(layer).__name__}'
            named[name] = layer
            relations[name] = prev
            prev = name
        relations[0] = prev
        super().__init__(layers=named, relations=relations, *args, **kwargs)


class HourglassFusion:
    """Whole-network inference kernel for the single-channel hourglass of make_paragraph
    (my_model/model.py:137-190): down_1, down_2 (conv 5x5 stride 2 + LeakyRelu), up_2, up_1
    (Upsample2D(2) + conv 5x5 + LeakyRelu), end (conv 5x5 + Sigmoid) as ONE launch of
    uocr_hourglass1_fwd; the intermediate maps never leave shared memory.

    Attached to the (flattened) top-level Model as `infer_fusion`; returns None (-> layer-by-layer
    plan) whenever the topology, the hyper-parameters or the input geometry are not the ones the
    kernel implements."""

    CHANNELS_1 = [(1, 1)] * 5                                     # make_paragraph: uocr_hourglass1_fwd
    CHANNELS_4 = [(1, 4), (4, 4), (4, 4), (4, 4), (4, 2)]         # make_line (my_model/model.py:194-248): uocr_hourglass4_fwd

    def __init__(self, prefix):
        p = prefix
        self._packed = None
        self.chain = [f'{p}/down_1/conv_1', f'{p}/down_1/leaky_relu_1',
                      f'{p}/down_2/conv_1', f'{p}/down_2/leaky_relu_1',
                      f'{p}/up_2/upsample', f'{p}/up_2/conv_block/conv_1', f'{p}/up_2/conv_block/leaky_relu_1',
                      f'{p}/up_1/upsample', f'{p}/up_1/conv_block/conv_1', f'{p}/up_1/conv_block/leaky_relu_1',
                      f'{p}/end/conv_1', f'{p}/end/sigmoid']

    @classmethod
    def detect(cls, model):
        """A HourglassFusion for `model` if its flattened layers are exactly the single-channel hourglass, else None."""
        tail = '/down_1/conv_1'
        for name in model.layers:
            if name.endswith(tail):
                fusion = cls(name[:-len(tail)])
                if fusion._blocks(model) is not None:
                    return fusion
        return None

    def _blocks(self, model):
        """[(conv, act)] in kernel order, or None if the network is not the expected hourglass."""
        if set(model.layers) != set(self.chain) or model.outputs_count != 1 or model.inputs_count != 1:
            return None
        prev = 0
        for name in self.chain:                              # a plain chain input -> ... -> output
            if list(model.relations[name]) != [prev]:
                return None
            prev = name
        if list(model.relations[0]) != [prev]:
            return None
        L = model.layers
        out = []
        for conv_i, act_i, ups_i, stride in ((0, 1, None, (2, 2)), (2, 3, None, (2, 2)), (5, 6, 4, (1, 1)),
                                             (8, 9, 7, (1, 1)), (10, 11, None, (1, 1))):
            conv, act = L[self.chain[conv_i]], L[self.chain[act_i]]
            if ups_i is not None:
                ups = L[self.chain[ups_i]]
                if type(ups) is not Upsample2D or ups.scale_factor != (2, 2):
                    return None
            if (type(conv) is not Convolutional2D or conv.kernel_size != (5, 5) or conv.padding != (2, 2)
                    or conv.stride != stride or conv.padding_value != 0 or not conv.bias):
                return None
            out.append((conv, act))
        channels = [(conv.in_channels, conv.out_channels) for conv, _ in out]
        if channels not in (self.CHANNELS_1, self.CHANNELS_4):
            return None
        return out

    def _applies(self, model, X):
        """(blocks, inner activations, end activation, four-channel) if the kernel takes `X`, else None."""
        blocks = self._blocks(model)
        if blocks is None:
            return None
        if len(X.shape) != 4 or X.shape[3] != 1 or X.shape[1] % 4 or X.shape[2] % 4 or X.shape[0] > 65535:
            return None
        inner = [_act_code(act) for _, act in blocks[:4]]
        end = _act_code(blocks[4][1])
        if (end is None or any(a is None or a[0] != ACT_LEAKY or a[1] > 1 for a in inner)
                or len({a[1] for a in inner}) != 1):
            return None
        four = blocks[1][0].in_channels == 4
        if four and CP.math_mode != MATH_TF32:             # the four-channel kernel is tensor-core (TF32) only
            return None
        return blocks, inner, end, four

    def _packed_image(self, blocks, wp):
        key = (CP.weights_generation, tuple(conv.w.value.ptr for conv, _ in blocks))
        if self._packed is None or self._packed[0] != key:         # tensor-core operand image of the five weight tensors
            count = ctypes.c_int64()
            lib.uocr_hourglass4_packed_floats(ctypes.byref(count))
            packed = DeviceArray((count.value,))
            lib.uocr_hourglass4_pack(wp, packed.ptr, stream())
            self._packed = (key, packed)
        return self._packed[1]

    def __call__(self, model, inputs, extents=None, extents_ptr=None):
        """`extents` (host (N, 2)) / `extents_ptr` (the same table on the device): a ragged batch (Model.predict_ragged),
        run by the four-channel kernel's ragged variant when every extent is a multiple of 4; None (-> the layer plan)
        for every other ragged case, since the one-channel kernel keeps its maps on chip where they cannot be masked."""
        X = as_device(inputs[0])
        found = self._applies(model, X)
        if found is None:
            return None
        blocks, inner, end, four = found
        if extents is not None and (not four or (np.asarray(extents) % 4).any()):
            return None
        n, h, w, _ = X.shape
        ptrs = ctypes.c_void_p * 5
        wp = ptrs(*[conv.w.value.ptr for conv, _ in blocks])
        bp = ptrs(*[conv.b.value.ptr for conv, _ in blocks])
        last = blocks[4][1]
        last.progress_tracker.start_tracking(last.name, 'forward')
        y = DeviceArray((n, h, w, blocks[4][0].out_channels))
        if extents is not None:
            lib.uocr_hourglass4_fwd_packed_ragged(X.ptr, self._packed_image(blocks, wp).ptr, bp, y.ptr, extents_ptr, n, h,
                                                  w, inner[0][1], end[0], end[1], stream())
        elif four:
            lib.uocr_hourglass4_fwd_packed(X.ptr, self._packed_image(blocks, wp).ptr, bp, y.ptr, n, h, w, inner[0][1],
                                           end[0], end[1], stream())
        else:
            lib.uocr_hourglass1_fwd_mode(X.ptr, wp, bp, y.ptr, n, h, w, inner[0][1], end[0], end[1], CP.math_mode, stream())
        last.progress_tracker.stop_tracking(last.name, 'forward')
        return [y]
