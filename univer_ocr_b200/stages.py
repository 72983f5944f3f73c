"""The crop stages between the sub-networks on the device (SURVEY.md 8f, row 4).

Mirrors `web_app/components/interpreter/interpreter.py` -- same class names, constructor arguments, call signatures and
result nesting -- with every array operation on the GPU:

    label_layer                       :16-22     glue.above_mean / glue.label_components / glue.label_stats
    rotate_array                      :188-192   uocr_rotate_f32 / uocr_rotate_nearest_u8   (ndimage.rotate, order 1 / 0)
    FindObjectHeightInRotated._func   :229-232   nearest rotation of the mask + uocr_mask_bbox
    CropAndRotateSingleParagraph      :295-343   masked crop, ternary search for the angle, rotation, crop
    CropAndRotateParagraphs           :346-374
    rearrange_lines                   :41-84     centres of mass from the device's label statistics, sorting on the host
    CropRotateAndZoomLines            :423-523   thresholded -> label -> rearrange -> crop, quarter turn, zoom, pad

What stays on the host is the control flow over objects (a handful of boxes and centres of mass per paragraph) -- the
reference spreads that over worker processes (`workers_count`), which has no counterpart here: the argument is accepted
and ignored.  Results are device arrays (`to_host=False`, default) or NumPy arrays like the reference's.

SciPy's resampling is reproduced bit for bit (tests/test_gpu_stages.py compares with scipy.ndimage on the same inputs);
`scipy.special.cosdg / sindg` give the rotation matrix exactly as ndimage.rotate builds it.
"""
import ctypes

import numpy as np

from . import glue
from ._lib import lib
from .nn.gpu import DeviceArray, as_device, stream


# ---------------------------------------------------------------------------------------------- resampling primitives

_special = None
_corners = {}


def rotate_geometry(h, w, angle):
    """Output plane shape, matrix and offset of `ndimage.rotate(..., axes=(2, 1), reshape=True)` for an (h, w) plane
    (scipy/ndimage/_interpolation.py: rotate): input (y, x) = matrix @ output (y, x) + offset.  The two matrix products
    stay NumPy's (`@`, i.e. the BLAS rounding SciPy itself gets); everything around them is scalar Python arithmetic
    -- the angle search calls this four times per step and 30 us of array bookkeeping per call was most of its time."""
    global _special
    if _special is None:
        from scipy import special as _special_module
        _special = _special_module
    c, s = float(_special.cosdg(angle)), float(_special.sindg(angle))
    m = np.array([[c, s], [-s, c]], dtype=np.float64)
    corners = _corners.get((h, w))
    if corners is None:
        corners = _corners[(h, w)] = np.array([[0, 0, h, h], [0, w, 0, w]], dtype=np.float64)
        if len(_corners) > 4096:
            _corners.clear()
    bounds = (m @ corners).tolist()
    # (np.ptp(out_bounds, axis=1) + 0.5).astype(int): max - min per row, + 0.5, truncated
    oh = int((max(bounds[0]) - min(bounds[0])) + 0.5)
    ow = int((max(bounds[1]) - min(bounds[1])) + 0.5)
    centre = (m @ np.array([(oh - 1) / 2, (ow - 1) / 2], dtype=np.float64)).tolist()
    offset = np.array([(h - 1) / 2 - centre[0], (w - 1) / 2 - centre[1]], dtype=np.float64)
    return (oh, ow), m, offset


def _device(array, dtype=None):
    if isinstance(array, DeviceArray):
        return array
    host = np.asarray(array)
    if host.dtype == np.bool_ or host.dtype == np.uint8 or dtype == np.uint8:
        return DeviceArray.from_host(np.ascontiguousarray(host, dtype=np.uint8), np.uint8)
    return as_device(np.ascontiguousarray(host, dtype=np.float32))


def rotate_array(array, angle=None, good_rotation=True):
    """interpreter.py:188-192 for an (N, H, W, C) device array: float32 (order 1, or 0 when not `good_rotation`) or a
    uint8 mask (nearest only -- the reference rotates masks with `good_rotation=False`)."""
    if angle is None:
        return array
    array = _device(array)
    n, h, w, c = array.shape
    (oh, ow), m, off = rotate_geometry(h, w, angle)
    out = DeviceArray.empty((n, oh, ow, c), array.dtype)
    mat = (ctypes.c_double * 4)(*m.ravel())
    offs = (ctypes.c_double * 2)(*off)
    if array.dtype == np.uint8:
        if good_rotation:
            raise TypeError('masks are rotated with good_rotation=False (nearest neighbour)')
        lib.uocr_rotate_nearest_u8(array.ptr, out.ptr, n, h, w, c, oh, ow, mat, offs, stream())
    else:
        lib.uocr_rotate_f32(array.ptr, out.ptr, n, h, w, c, oh, ow, mat, offs, 1 if good_rotation else 0, stream())
    return out


def mask_bbox(mask):
    """`ndimage.find_objects(mask)[0]` of a boolean (N, H, W, C) device array -> (slice_y, slice_x); IndexError when the
    mask is empty (the reference indexes an empty list there)."""
    n, h, w, c = mask.shape
    box = DeviceArray.empty((4,), np.int32)
    lib.uocr_mask_bbox(mask.ptr, box.ptr, n, h, w, c, stream())
    y0, y1, x0, x1 = (int(v) for v in box.get())
    if y1 < 0:
        raise IndexError('list index out of range')           # find_objects(all-False)[0]
    return slice(y0, y1 + 1), slice(x0, x1 + 1)


def crop(array, region_y, region_x, labels=None, label=0):
    """`array[:, region_y, region_x, :]`, or `(array * (labels == label))[:, region_y, region_x, :]`."""
    n, h, w, c = array.shape
    ch, cw = region_y.stop - region_y.start, region_x.stop - region_x.start
    out = DeviceArray.empty((n, ch, cw, c), np.float32)
    lib.uocr_crop_masked_f32(array.ptr, labels.ptr if labels is not None else None, label, out.ptr, n, h, w, c,
                             region_y.start, region_x.start, ch, cw, stream())
    return out


def crop_label_mask(labels, label, region_y, region_x):
    """`(labels == label)[:, region_y, region_x, :]` as a uint8 (N, h, w, 1) mask."""
    n, h, w = labels.shape[:3]
    ch, cw = region_y.stop - region_y.start, region_x.stop - region_x.start
    out = DeviceArray.empty((n, ch, cw, 1), np.uint8)
    lib.uocr_crop_label_mask(labels.ptr, label, out.ptr, n, h, w, region_y.start, region_x.start, ch, cw, stream())
    return out


def zoom_nearest(array, zoom, minimal_width=None):
    """`ndimage.zoom(array, (1, zoom, zoom, 1), order=0)` followed by the zero padding to `minimal_width` columns
    (CropRotateAndZoomLines._func2, :513-521)."""
    n, h, w, c = array.shape
    oh, ow = int(round(h * zoom)), int(round(w * zoom))
    owp = max(ow, minimal_width) if minimal_width is not None else ow
    out = DeviceArray.empty((n, oh, owp, c), np.float32)
    lib.uocr_zoom_nearest_f32(array.ptr, out.ptr, n, h, w, c, oh, ow, owp, stream())
    return out


def label_objects(mask):
    """label_layer (:16-22) on the device: labels (N, H, W, 1) int32 + per-object statistics of image 0
    (`glue.label_stats`).  `mask`: a uint8 / boolean mask (foreground = above its mean) or a float32 map."""
    mask = _device(mask)
    if mask.dtype != np.uint8:
        mask = glue.above_mean(mask)
    labels, counts = glue.label_components(mask)
    return labels, glue.label_stats(labels, counts)[0]


# ---------------------------------------------------------------------------------------------- paragraphs

def rotated_height(mask, angle):
    """FindObjectHeightInRotated._func (:229-232)."""
    region_y, _ = mask_bbox(rotate_array(mask, angle, good_rotation=False))
    return region_y.stop - region_y.start


def rotated_heights(mask, angles):
    """`rotated_height` for one or two angles in one launch: the rows each nearest rotation would span, read off the
    source mask without materialising the rotated copies (uocr_rotated_row_spans)."""
    k = len(angles)
    spans = DeviceArray.empty((2 * k,), np.int32)
    _launch_row_spans(mask, angles, spans, 0)
    host = spans.get()
    if (host[1::2] < 0).any():
        raise IndexError('list index out of range')           # find_objects(all-False)[0]
    return [int(host[2 * i + 1] - host[2 * i] + 1) for i in range(k)]


def _launch_row_spans(mask, angles, spans, slot, reset=True):
    """Queues uocr_rotated_row_spans for `angles` (1 or 2) of `mask` into spans[slot : slot + 2 * len(angles)]."""
    n, h, w, c = mask.shape
    k = len(angles)
    geoms = [rotate_geometry(h, w, angle) for angle in angles]
    mats = (ctypes.c_double * (4 * k))(*[v for _, m, _ in geoms for v in m.ravel()])
    offs = (ctypes.c_double * (2 * k))(*[v for _, _, off in geoms for v in off])
    shapes = (ctypes.c_int64 * (2 * k))(*[v for shape, _, _ in geoms for v in shape])
    lib.uocr_rotated_row_spans(mask.ptr, spans.ptr + 4 * slot, n, h, w, c, k, mats, offs, shapes, 1 if reset else 0,
                               stream())


def find_rotation_angles(masks, EPS=1.0):
    """The ternary search of CropAndRotateSingleParagraph._func (:318-333) for several paragraph masks in lockstep: the
    angle in (0, 180) at which each nearest-rotated mask spans the fewest rows; None within EPS of 0 / 180.  Every mask
    takes the same number of steps (the interval shrinks by a third per step whatever the comparison says), so one step
    is one launch per mask (both probe angles, `uocr_rotated_row_spans`) and ONE read-back for all of them."""
    low, high = [0.0] * len(masks), [180.0] * len(masks)
    steps, width = 0, 180.0
    while width > EPS:                                        # every mask takes the same number of steps
        width, steps = width - width / 3, steps + 1          # (an upper bound is enough: the table is only sized by it)
    steps += 2
    per_step = 4 * max(len(masks), 1)
    table = DeviceArray.empty((steps * per_step,), np.int32)
    lib.uocr_row_spans_reset(table.ptr, steps * per_step // 2, stream())
    host = np.empty(per_step, np.int32)
    step = 0
    while masks and high[0] - low[0] > EPS:
        assert step < steps
        probes = []
        for i, mask in enumerate(masks):
            a = low[i] + (high[i] - low[i]) / 3
            b = high[i] - (high[i] - low[i]) / 3
            probes.append((a, b))
            _launch_row_spans(mask, (a, b), table, step * per_step + 4 * i, reset=False)
        lib.uocr_memcpy_d2h(host.ctypes.data, table.ptr + 4 * step * per_step, host.nbytes, stream())
        lib.uocr_stream_sync(stream())
        step += 1
        for i, (a, b) in enumerate(probes):
            y0a, y1a, y0b, y1b = (int(v) for v in host[4 * i:4 * i + 4])
            if y1a < 0 or y1b < 0:
                raise IndexError('list index out of range')       # find_objects(all-False)[0]
            if y1a - y0a < y1b - y0b:
                high[i] = b
            else:
                low[i] = a
    angles = [(h + l) / 2 for l, h in zip(low, high)]
    return [angle if EPS <= angle <= 180.0 - EPS else None for angle in angles]


def find_rotation_angle(mask, EPS=1.0):
    return find_rotation_angles([mask], EPS)[0]


class CropAndRotateParagraphs:
    """interpreter.py:346-374 (with CropAndRotateSingleParagraph, :234-343):

        result = CropAndRotateParagraphs(workers_count, find_rotation)(masks, images)
        result[image_id][paragraph_id]      # (1, h, w, C): the paragraph, masked, straightened, cropped

    `masks`: the Paragraph prediction (1, H, W, 1); `images`: list of (1, H, W, C) maps to cut."""

    def __init__(self, workers_count=None, find_rotation=True, EPS=1.0, to_host=False):
        self.workers_count, self.find_rotation, self.EPS, self.to_host = workers_count, find_rotation, EPS, to_host
        self.angles = []                                       # of the last call, per paragraph (None: not rotated)

    def __call__(self, masks, images):
        images = [_device(image) for image in images]
        labels, objects = label_objects(masks)
        cut = self.cut(labels, objects, images)
        self.angles = self.search_angles([cut])[0]
        return self.straighten(cut, self.angles, len(images))

    # The three phases of a call, also run by predict.TextPipeline.batch over the paragraphs of many pages at once.
    @staticmethod
    def cut(labels, objects, images):
        """Per paragraph of a (1, H, W, 1) label map and its `glue.label_stats` objects: the object's mask and the masked
        maps, cut to its box (CropAndRotateSingleParagraph._run, :300-309)."""
        cut = []
        for paragraph_id, obj in enumerate(objects):
            region_y, region_x = obj['slices']
            mask = crop_label_mask(labels, paragraph_id + 1, region_y, region_x)
            cut.append((mask, [crop(image, region_y, region_x, labels, paragraph_id + 1) for image in images]))
        return cut

    def search_angles(self, cuts):
        """._func (:312-343), first part: the angle of every paragraph of every `cut` result, all searched in lockstep."""
        masks = [mask for cut in cuts for mask, _ in cut]
        angles = find_rotation_angles(masks, self.EPS) if self.find_rotation else [None] * len(masks)
        out, pos = [], 0
        for cut in cuts:
            out.append(angles[pos:pos + len(cut)])
            pos += len(cut)
        return out

    def straighten(self, cut, angles, image_count):
        """._func, second part: the rotated mask's box, the rotated maps cut to it -> result[image_id][paragraph_id]."""
        result = [[None for _ in cut] for _ in range(image_count)]
        for paragraph_id, ((mask, arrays), angle) in enumerate(zip(cut, angles)):
            out_y, out_x = mask_bbox(rotate_array(mask, angle, good_rotation=False))
            for image_id, arr in enumerate(arrays):
                res = crop(rotate_array(arr, angle), out_y, out_x)
                result[image_id][paragraph_id] = res.get() if self.to_host else res
        return result


# ---------------------------------------------------------------------------------------------- lines

def rearrange_lines(top, bottom, h, w):
    """interpreter.py:41-84 on object tables instead of object masks: `top` / `bottom` are the `glue.label_stats`
    entries of the two line-mask channels of one paragraph (h x w).  -> (top objects, bottom objects, rotation):
    every top object paired with the nearest bottom object, both sorted along the reading direction.  Centres of mass
    are the 4-vectors (0, y, x, 0) `ndimage.center_of_mass` returns for a (1, h, w, 1) mask."""
    def cm(objs):
        return [(np.array((0.0, o['center_of_mass'][0], o['center_of_mass'][1], 0.0)), o) for o in objs]

    tops, bottoms = cm(top), cm(bottom)
    paired = [sorted(bottoms, key=lambda x: np.linalg.norm(c[0] - x[0]))[0][1] for c in tops]
    dist_point = tops[0][0] - bottoms[0][0]                    # IndexError without objects, like the reference
    while 0 < dist_point[1] < h or 0 < dist_point[2] < w:
        dist_point *= 1000
    sort_key = rotation = None
    if abs(dist_point[1]) > abs(dist_point[2]):
        if dist_point[1] < 0:
            sort_key, rotation = (lambda x: x[0][1]), None
        elif dist_point[1] > h:
            sort_key, rotation = (lambda x: -x[0][1]), 180
    else:
        if dist_point[2] < 0:
            sort_key, rotation = (lambda x: x[0][2]), 270
        elif dist_point[2] > w:
            sort_key, rotation = (lambda x: -x[0][2]), 90
    if sort_key is None:                                       # the reference leaves `sort_key` unbound here
        raise UnboundLocalError("cannot access local variable 'sort_key' where it is not associated with a value")
    tops, bottoms = cm(top), cm(paired)
    return [t[1] for t in sorted(tops, key=sort_key)], [b[1] for b in sorted(bottoms, key=sort_key)], rotation


def line_region(top_obj, bottom_obj):
    """CropRotateAndZoomLines._func1 (:493-501): the box around a line's top and bottom marks."""
    (ty, tx), (by, bx) = top_obj['slices'], bottom_obj['slices']
    return (slice(min(ty.start, by.start), max(ty.stop, by.stop)),
            slice(min(tx.start, bx.start), max(tx.stop, bx.stop)))


def crop_rotate_zoom(image, y, x, rotation, zoomed_height, minimal_width):
    """CropRotateAndZoomLines._func2 (:503-523)."""
    final = crop(image, y, x)
    if rotation is not None:
        final = rotate_array(final, rotation)
    if zoomed_height is not None:
        final = zoom_nearest(final, zoomed_height / final.shape[1], minimal_width)
    elif minimal_width is not None and final.shape[2] < minimal_width:
        final = zoom_nearest(final, 1.0, minimal_width)        # zoom 1 = copy; pads the width
    return final


class CropRotateAndZoomLines:
    """interpreter.py:423-491:

        result = CropRotateAndZoomLines(workers_count, zoomed_height, minimal_width)(masks, arrays)
        result[array_id][paragraph_id][line_id]      # (1, zoomed_height, >= minimal_width, C)

    `masks[paragraph_id]`: the Line prediction (1, h, w, 2) of a cropped paragraph (channel 0: top marks, 1: bottom
    marks); `arrays[array_id][paragraph_id]`: the (1, h, w, C) maps to cut lines from."""

    def __init__(self, workers_count=None, zoomed_height=None, minimal_width=None, to_host=False):
        self.workers_count, self.zoomed_height, self.minimal_width = workers_count, zoomed_height, minimal_width
        self.to_host = to_host

    def __call__(self, masks, arrays):
        result = [[] for _ in arrays]
        for paragraph_id, mask in enumerate(masks):
            mask = _device(mask)
            _, h, w, _ = mask.shape
            marks = glue.thresholded(mask)                     # per channel: arr > 0.5 * (mean + max)
            # label_layer(top), label_layer(bottom): the two channels as two images of one labelling call
            top, bottom = glue.label_stats(*glue.label_components(glue.channel_planes(marks)))
            tops, bottoms, rotation = rearrange_lines(top, bottom, h, w)
            for array_id in range(len(arrays)):
                result[array_id].append([])
            for top_obj, bottom_obj in zip(tops, bottoms):
                y, x = line_region(top_obj, bottom_obj)
                for array_id in range(len(arrays)):
                    image = _device(arrays[array_id][paragraph_id])
                    line = crop_rotate_zoom(image, y, x, rotation, self.zoomed_height, self.minimal_width)
                    result[array_id][paragraph_id].append(line.get() if self.to_host else line)
        return result
