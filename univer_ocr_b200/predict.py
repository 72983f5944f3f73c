"""The reference's PREDICT pipeline on the device (SURVEY.md 8f, rows 3 and 4): `PageStage` (its first stage, batched over
pages) and `TextPipeline` (the whole model system of `my_model/model.py:688-717` for one page, page -> text).

Reference (`my_model/predict.py:12-23`, `my_model/model.py:695-699`): load `model_weights.json`, pad the page to a
multiple of 16 (`make_divisible_by`), run Monochrome, feed its prediction to Paragraph, move BOTH float64 maps to the
host, where `CropAndRotateParagraphs` starts by binarising the paragraph map (`interpreter/interpreter.py:437-447`).
Here the padding, the two networks (Monochrome conv pair on tcgen05, Paragraph as one fused kernel) and the binarisation
and the connected-component labelling of that mask (`label_layer`, `interpreter/interpreter.py:16-22`) run back to
back on the device; what the crop stage needs crosses the host link as one float32 map + a uint8 mask or an int32
label map (5-8 bytes per pixel instead of 16).  `TextPipeline` continues on the device through the crop stages
(`stages.py`), Line, Char and PredToText.
"""
import ctypes

import numpy as np

from . import glue, my_model, weights_io
from ._lib import lib
from .nn.gpu import CP, DeviceArray, as_device, concatenate, stream


class PageStage:
    """
        stage = PageStage(weights_path='model_weights.json')
        out = stage(pages)                      # pages: (N, H, W, 1) host or device array, any H, W
        host = stage.to_host(out)               # {'monochrome_pred': float32, 'paragraph_mask': uint8, ...}

    Networks are (re)built per padded page shape and cached; weights come from the JSON file (or stay at their
    initialisation when the file is missing, like the reference)."""

    def __init__(self, weights_path=None, divisor=(16, 16)):
        CP.use_gpu()
        self.weights_path, self.divisor = weights_path, divisor
        self._weights = weights_io.read(weights_path) if weights_path is not None else {}
        self._models = {}

    def models_for(self, shape):
        shape = tuple(shape)
        if shape not in self._models:
            mono, para = my_model.make_monochrome(shape), my_model.make_paragraph(shape)
            for model in (mono, para):
                model.set_weights(self._weights)
            self._models[shape] = (mono, para)
        return self._models[shape]

    def __call__(self, pages):
        x = glue.make_divisible_by(as_device(pages), *self.divisor)
        mono, para = self.models_for(x.shape)
        monochrome_pred = mono.predict(x)[0]
        paragraph_pred = para.predict(monochrome_pred)[0]
        paragraph_mask = glue.thresholded(paragraph_pred)
        # what CropAndRotateParagraphs does first with that mask (interpreter/interpreter.py:437-447 -> label_layer :16-22)
        paragraph_labels, paragraph_count = glue.label_components(paragraph_mask)
        return {'padded': x, 'monochrome_pred': monochrome_pred, 'paragraph_pred': paragraph_pred,
                'paragraph_mask': paragraph_mask, 'paragraph_labels': paragraph_labels,
                'paragraph_count': paragraph_count}

    @staticmethod
    def to_host(result, want=('monochrome_pred', 'paragraph_mask')):
        return {key: np.asarray(result[key].get()) for key in want}


class TextPipeline:
    """The reference's PREDICT model system (`my_model/model.py:688-717`) with every stage on the device:

        page -> pad to a multiple of 16 -> Monochrome -> Paragraph
             -> CropAndRotateParagraphs(paragraph_pred, [monochrome_pred])      (ParagraphCrop, :551-575)
             -> pad every paragraph to a multiple of 16 -> Line per paragraph    (LineSelector, :353-372)
             -> CropRotateAndZoomLines(CHAR_INPUT_HEIGHT, CHAR_FIXED_WIDTH)      (LineCrop, :595-612)
             -> Char per line                                                   (CharSelector, :375-400)
             -> PredToText                                                      (:648-657)

        pipe = TextPipeline('model_weights.json', chars=CHARS, are_similar=are_similar)
        out = pipe(page)                  # page: (1, H, W, 1) host or device array
        out['text'][paragraph_id][line_id]
        outs = pipe.batch(pages)          # list of (1, H, W, 1) arrays of any sizes, or one (N, H, W, 1) array
        outs[page_id]['text'][paragraph_id][line_id]

    Nothing but the final hit tables (1 byte per score) and the stages' object tables (a few numbers per paragraph / line)
    crosses the host link; the reference moves every map to the host and back between the stages (`move_from_gpu_*`,
    `move_to_gpu_*`).  Each network is built once and runs every input shape, weights from the JSON file.  `predictors` replaces networks by callables `DeviceArray -> DeviceArray` (tests, or models kept
    elsewhere); without `chars` / `are_similar` (the reference's `primitives.CHARS`, `are_similar`) the text is returned
    as lists of class ids."""

    NETWORKS = ('monochrome', 'paragraph', 'line', 'char')

    def __init__(self, weights_path=None, find_rotation=True, predictors=None, chars=None, are_similar=None,
                 divisor=(16, 16)):
        from . import stages
        CP.use_gpu()
        self.divisor, self.chars, self.are_similar = divisor, chars, are_similar
        self._weights = weights_io.read(weights_path) if weights_path is not None else {}
        self._models, self.predictors = {}, dict(predictors or {})
        self.crop_paragraphs = stages.CropAndRotateParagraphs(None, find_rotation)
        self.crop_lines = stages.CropRotateAndZoomLines(None, my_model.CHAR_INPUT_HEIGHT, my_model.CHAR_FIXED_WIDTH)

    def model(self, name, shape):
        """The pipeline's one instance of network `name`, built for the first input shape it sees.  Every network's
        parameters, fusion plans and cached kernel operands are independent of the input's H, W and batch, so the same
        instance runs every crop: the weights are uploaded once, and every crop is read by the same network."""
        if name not in self._models:
            model = my_model.MAKERS[name](tuple(shape))
            model.set_weights(self._weights)
            self._models[name] = model
        return self._models[name]

    def predict(self, name, x):
        if name in self.predictors:
            return self.predictors[name](x)
        return self.model(name, x.shape).predict(x)[0]

    def to_text(self, char_pred):
        return self._hits_text(glue.row_max_hits(char_pred).get())

    def __call__(self, page):
        x = glue.make_divisible_by(as_device(page), *self.divisor)
        monochrome_pred = self.predict('monochrome', x)
        paragraph_pred = self.predict('paragraph', monochrome_pred)
        cropped = self.crop_paragraphs(paragraph_pred, [monochrome_pred])[0]
        cropped = [glue.make_divisible_by(t, *self.divisor) for t in cropped]
        line_pred = [self.predict('line', t) for t in cropped]
        lines = self.crop_lines(line_pred, [cropped])[0]
        char_pred = [[self.predict('char', line) for line in paragraph] for paragraph in lines]
        text = [[self.to_text(pred) for pred in paragraph] for paragraph in char_pred]
        return {'text': text, 'angles': list(self.crop_paragraphs.angles), 'monochrome_pred': monochrome_pred,
                'paragraph_pred': paragraph_pred, 'cropped_monochrome': cropped, 'line_pred': line_pred,
                'cropped_2_monochrome': lines, 'char_pred': char_pred}

    # ---- batches of pages -------------------------------------------------------------------------------------------
    CHAR_WIDTH_MULTIPLE = 8              # the Char canvas width is the widest line rounded up to this

    def _run_each(self, name, xs):
        """Stand-in `name` called once per item, as in `__call__`."""
        return [self.predictors[name](x) for x in xs]

    def _ragged(self, name, items, width_multiple=1):
        """Network `name` once over `items` ((1, h_i, w_i, C) device arrays) packed into one zero-filled canvas ->
        (output canvas, output extents, input extents) of Model.predict_ragged."""
        ext = np.array([x.shape[1:3] for x in items], dtype=np.int64)
        c = items[0].shape[3]
        h = int(ext[:, 0].max())
        w = -(-int(ext[:, 1].max()) // width_multiple) * width_multiple
        model = self.model(name, (len(items), h, w, c))
        dev_ext = DeviceArray.from_host(ext.astype(np.int32), np.int32)
        canvas = DeviceArray.empty((len(items), h, w, c))
        srcs = (ctypes.c_void_p * len(items))(*[x.ptr for x in items])
        lib.uocr_pack_hw_f32(srcs, dev_ext.ptr, canvas.ptr, len(items), h, w, c, stream())
        outs, out_ext = model.predict_ragged(canvas, ext)
        return outs[0], out_ext[0]

    def _unpack(self, canvas, ext):
        """Image i of a ragged output canvas -> its own (1, h_i, w_i, C) array, one launch for all."""
        n, h, w, c = canvas.shape
        dsts = [DeviceArray.empty((1, int(eh), int(ew), c)) for eh, ew in ext]
        ptrs = (ctypes.c_void_p * n)(*[d.ptr for d in dsts])
        dev_ext = DeviceArray.from_host(np.asarray(ext, np.int32), np.int32)
        lib.uocr_unpack_hw_f32(canvas.ptr, dev_ext.ptr, ptrs, n, h, w, c, stream())
        return dsts

    def batch(self, pages):
        """`__call__` for many pages: `pages` is a list of (1, H, W, 1) arrays of any sizes or one (N, H, W, 1) array.
        -> one dict per page with the keys and nesting `__call__` returns.  Monochrome -> Paragraph run once per distinct
        page size (the existing fused kernels), the paragraphs of all pages are labelled per page size and searched for
        their angles in lockstep, then Line runs ONCE over all paragraphs and Char ONCE over all lines, each on a ragged
        batch (Model.predict_ragged), and one hit table is read back for all lines.  Stand-ins from `predictors` are
        called once per item, as in `__call__`."""
        if isinstance(pages, (list, tuple)):
            pages = [as_device(p) for p in pages]
        else:
            whole = as_device(pages)
            pages = [whole[i:i + 1] for i in range(whole.shape[0])]
        for p in pages:
            if len(p.shape) != 4 or p.shape[0] != 1 or p.shape[3] != 1:
                raise ValueError(f'a page is (1, H, W, 1), got {p.shape}')
        n_pages = len(pages)
        mono, para, cut = [None] * n_pages, [None] * n_pages, [None] * n_pages
        groups = {}
        for i, p in enumerate(pages):
            groups.setdefault(tuple(p.shape[1:3]), []).append(i)
        # 1-2. pad, Monochrome -> Paragraph per page size; label the paragraphs of all pages of that size in one call
        for ids in groups.values():
            x = glue.make_divisible_by(concatenate([pages[i] for i in ids], axis=0), *self.divisor)
            if 'monochrome' in self.predictors:
                m = concatenate(self._run_each('monochrome', [x[k:k + 1] for k in range(len(ids))]), axis=0)
            else:
                m = self.predict('monochrome', x)
            if 'paragraph' in self.predictors:
                q = concatenate(self._run_each('paragraph', [m[k:k + 1] for k in range(len(ids))]), axis=0)
            else:
                q = self.predict('paragraph', m)
            labels, counts = glue.label_components(glue.above_mean(q))
            objects = glue.label_stats(labels, counts)
            for k, i in enumerate(ids):
                mono[i], para[i] = m[k:k + 1], q[k:k + 1]
                cut[i] = self.crop_paragraphs.cut(labels[k:k + 1], objects[k], [mono[i]])
        angles = self.crop_paragraphs.search_angles(cut)
        cropped = [[glue.make_divisible_by(t, *self.divisor) for t in self.crop_paragraphs.straighten(c, a, 1)[0]]
                   for c, a in zip(cut, angles)]
        # 3. Line once over every paragraph of every page
        flat = [t for page in cropped for t in page]
        if not flat:
            line_flat = []
        elif 'line' in self.predictors:
            line_flat = self._run_each('line', flat)
        else:
            line_flat = self._unpack(*self._ragged('line', flat))
        line_pred, pos = [], 0
        for page in cropped:
            line_pred.append(line_flat[pos:pos + len(page)])
            pos += len(page)
        lines = [self.crop_lines(lp, [cp])[0] for lp, cp in zip(line_pred, cropped)]
        # 4. Char once over every line of every page; one hit table for all of them
        all_lines = [line for page in lines for paragraph in page for line in paragraph]
        if not all_lines:
            preds, hits, rows = [], None, []
        elif 'char' in self.predictors:
            preds = self._run_each('char', all_lines)
            hits, rows = None, []
        else:
            out, rows = self._ragged('char', all_lines, self.CHAR_WIDTH_MULTIPLE)
            preds = [out[int(a):int(b)] for a, b in rows]
            hits = glue.row_max_hits(out).get()
        texts = []
        for k, pred in enumerate(preds):
            texts.append(self.to_text(pred) if hits is None else self._hits_text(hits[int(rows[k][0]):int(rows[k][1])]))
        results, pos = [], 0
        for i in range(n_pages):
            char_pred, text = [], []
            for paragraph in lines[i]:
                char_pred.append(preds[pos:pos + len(paragraph)])
                text.append(texts[pos:pos + len(paragraph)])
                pos += len(paragraph)
            results.append({'text': text, 'angles': list(angles[i]), 'monochrome_pred': mono[i],
                            'paragraph_pred': para[i], 'cropped_monochrome': cropped[i], 'line_pred': line_pred[i],
                            'cropped_2_monochrome': lines[i], 'char_pred': char_pred})
        return results

    def _hits_text(self, hits):
        if self.chars is not None and self.are_similar is not None:
            return glue.hits_to_text(hits, self.chars, self.are_similar)
        rows, cols = np.nonzero(hits)
        return [int(c) for c in cols[np.argsort(rows, kind='stable')]]
