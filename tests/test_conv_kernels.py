"""Bit-exact oracle tests of every convolution kernel variant, each row pinned to the kernel it must reach.

Every operand is a small integer (x, dy, w in {-2..2}, b in {-4..4}, padding_value in {0, 0.5, -1}, LeakyRelu slope
0.25), so every product and partial sum is a multiple of 0.25 below 2^22: FP32 represents it exactly, in any summation
order, and so do the TF32 operands of the tensor-core kernels (integers up to 2^11) with their FP32 accumulation.  A
correct kernel therefore equals the float64 oracle (oracle/np_oracle.py) BIT FOR BIT however large its reduction, and a
kernel that drops a pixel, repeats a tap or fills the border with the wrong value fails.  Each row asserts that the
oracle evaluated on |x|, |w|, |b|, |dy| stays <= 2^22, so a later edit cannot leave the exact regime unnoticed.  Sigmoid
epilogues are the one inexact step; they keep the FP32 tolerance of test_gpu_parity (rtol 1e-4 + 2e-6 max).

The TF32 kernels that read one operand from tensor memory (conv_row_tc.cu, conv_pair_tc.cu, conv_pair_rows_tc.cu) scale
their weights by (1 + 2^-11) before rounding them to TF32, to make the tensor core's truncation of the other operand
unbiased on real data.  Integers lose nothing to that truncation, so the scaling shows up as a 2^-10 relative offset;
their rows compare bit for bit with the oracle evaluated on those same operands (tc_scaled, trunc_tf32).

The rows call the C ABI directly (uocr_conv2d_fwd / _dgrad / _wgrad, uocr_conv3x3_pair_fwd / _bwd / _bwd_mode) and name
the kernel instantiation the dispatch must pick for them; test_each_row_reaches_its_kernel records the launched kernels
with torch.profiler and checks those names.  Rows whose id ends in `_unaligned` repeat a fast-kernel row on tensor views
offset by one float, which every fast path declines: the general kernels then give a second, independent result.
"""
import ctypes
import zlib

import numpy as np
import pytest

from oracle import np_oracle as O

pytestmark = pytest.mark.gpu

NONE, LEAKY, SIGMOID = 0, 1, 2
FP32, TF32 = 0, 1
ALPHA = 0.25
EXACT_LIMIT = 2.0 ** 22


@pytest.fixture(scope='module')
def nn():
    import univer_ocr_b200.nn as nn_
    nn_.CP.use_gpu()
    return nn_


# ------------------------------------------------------------------------------------------------ the table
class Row:
    """One call of uocr_conv2d_fwd / _dgrad / _wgrad.  (h, w) is the LOGICAL input size (the stored x is (h, w) / ups);
    `shift` names the tensors passed as views offset by one float; `kernels` are the demangled kernel names (whitespace
    ignored) the call must launch; kernels=None: the call must fail and leave its outputs untouched."""

    def __init__(self, id, op, n, h, w, cin, cout, k, p=0, s=1, pv=0.0, ups=1, mode=FP32, shift=(), kernels=()):
        self.id, self.op, self.n, self.h, self.w, self.cin, self.cout = id, op, n, h, w, cin, cout
        self.kh, self.kw = (k, k) if isinstance(k, int) else k
        self.ph, self.pw = (p, p) if isinstance(p, int) else p
        self.sh, self.sw = (s, s) if isinstance(s, int) else s
        self.pv, self.ups, self.mode, self.shift = pv, ups, mode, tuple(shift)
        self.kernels = None if kernels is None else tuple(kernels)

    @property
    def ho(self):
        return (self.h + 2 * self.ph - self.kh) // self.sh + 1

    @property
    def wo(self):
        return (self.w + 2 * self.pw - self.kw) // self.sw + 1

    def desc(self):
        from univer_ocr_b200._lib import ConvDesc
        return ConvDesc(self.n, self.h, self.w, self.cin, self.cout, self.kh, self.kw, self.ph, self.pw, self.sh,
                        self.sw, self.pv, 1, self.mode, self.ups)

    def unaligned(self, kernel):
        """The same call on tensor views offset by one float: the general kernel `kernel` must run."""
        return Row(self.id + '_unaligned', self.op, self.n, self.h, self.w, self.cin, self.cout, (self.kh, self.kw),
                   (self.ph, self.pw), (self.sh, self.sw), self.pv, self.ups, self.mode,
                   ('x', 'w', 'b', 'y', 'dy', 'dx'), None if kernel is None else [kernel])


def _fwd(*a, **k):
    return Row(a[0], 'fwd', *a[1:], **k)


def _dgrad(*a, **k):
    return Row(a[0], 'dgrad', *a[1:], **k)


def _wgrad(*a, **k):
    return Row(a[0], 'wgrad', *a[1:], **k)


def small_fwd(kh, kw, sh, sw, cin, cot, px, ups=1):
    return f'conv_small_fwd_kernel<{kh},{kw},{sh},{sw},{cin},{cot},{px},{ups}>'


def c1_fwd(kh, kw, sh, sw, cot, ups=1):
    return f'conv_c1_fwd_kernel<{kh},{kw},{sh},{sw},{cot},4,{ups},{32 if sh == 1 else 16}>'


def small_wgrad(*t):
    return 'conv_small_wgrad_kernel<' + ','.join(str(v) for v in t) + '>'


def fwd_direct(cout):
    return f'conv_fwd_direct_kernel<{next(c for c in (16, 8, 4, 2, 1) if cout % c == 0)}>'


def dgrad_direct(cin):
    return f'conv_dgrad_direct_kernel<{next(c for c in (8, 4, 2, 1) if cin % c == 0)}>'


def wgrad_tile(cout):
    return ('conv_wgrad_tile_kernel<64,64,4,4>' if cout >= 32 else
            'conv_wgrad_tile_kernel<64,16,4,1>' if cout >= 9 else 'conv_wgrad_tile_kernel<32,8,1,1>')


FINALIZE = 'conv_small_wgrad_finalize_kernel'
FLIP = 'flip_transpose_kernel'

ROWS = [
    # ---------------------------------------------------------------- forward, FP32 mode (conv_fast.cu, conv.cu)
    _fwd('c55_tile', 2, 45, 132, 1, 1, 5, 2, kernels=['conv55_c1_tile_kernel']),
    _fwd('c55_ups_tile', 2, 46, 136, 1, 1, 5, 2, ups=2, kernels=['conv55_c1_ups_tile_kernel']),
    _fwd('c1_55s1_w70', 2, 37, 70, 1, 1, 5, 2, kernels=[c1_fwd(5, 5, 1, 1, 1)]),
    _fwd('c1_55s1_pv05', 1, 37, 136, 1, 1, 5, 2, pv=0.5, kernels=[c1_fwd(5, 5, 1, 1, 1)]),
    _fwd('c1_55s1_p1', 1, 33, 68, 1, 1, 5, 1, kernels=[c1_fwd(5, 5, 1, 1, 1)]),
    _fwd('c1_55s1_p3', 1, 33, 68, 1, 1, 5, 3, pv=-1.0, kernels=[c1_fwd(5, 5, 1, 1, 1)]),
    _fwd('c1_55s1_ups_pv', 1, 34, 70, 1, 1, 5, 2, pv=0.5, ups=2, kernels=[c1_fwd(5, 5, 1, 1, 1, ups=2)]),
    _fwd('c1_55s2_1', 2, 37, 150, 1, 1, 5, 2, 2, pv=0.5, kernels=[c1_fwd(5, 5, 2, 2, 1)]),
    _fwd('c1_55s2_4', 2, 36, 300, 1, 4, 5, 2, 2, kernels=[c1_fwd(5, 5, 2, 2, 4)]),
    _fwd('c1_55s2_8', 1, 35, 140, 1, 8, 5, (1, 3), 2, pv=-1.0, kernels=[c1_fwd(5, 5, 2, 2, 4)]),
    _fwd('c1_33_16_p0', 2, 35, 130, 1, 16, 3, 0, kernels=[c1_fwd(3, 3, 1, 1, 16)]),
    _fwd('c1_33_16_p1', 2, 35, 131, 1, 16, 3, 1, pv=0.5, kernels=[c1_fwd(3, 3, 1, 1, 16)]),
    _fwd('c1_33_32_p2', 1, 33, 60, 1, 32, 3, 2, kernels=[c1_fwd(3, 3, 1, 1, 16)]),
    _fwd('c1_53_16_ph0', 2, 37, 140, 1, 16, (5, 3), (0, 1), (2, 1), kernels=[c1_fwd(5, 3, 2, 1, 16)]),
    _fwd('c1_53_128_ph2', 1, 36, 70, 1, 128, (5, 3), (2, 1), (2, 1), pv=0.5, kernels=[c1_fwd(5, 3, 2, 1, 16)]),
    _fwd('c1_53_64_wshift', 2, 21, 150, 1, 64, (5, 3), (0, 1), (2, 1), shift=('w',), kernels=[c1_fwd(5, 3, 2, 1, 16)]),
    _fwd('wide64', 2, 21, 150, 1, 64, (5, 3), (0, 1), (2, 1), kernels=['conv_c1_wide64_kernel<5,3,2,1,7>']),
    _fwd('wide64_pv', 1, 34, 260, 1, 64, (5, 3), (2, 1), (2, 1), pv=0.5, kernels=['conv_c1_wide64_kernel<5,3,2,1,7>']),
    # Cin = 1 past the grid limits of the shared-tile kernels (grid z = N * Cout / COT > 65535)
    _fwd('small_c1_33_16', 65537, 2, 4, 1, 16, 3, 1, kernels=[small_fwd(3, 3, 1, 1, 1, 16, 4)]),
    _fwd('small_c1_55s1', 65537, 4, 8, 1, 1, 5, 2, kernels=[small_fwd(5, 5, 1, 1, 1, 1, 8)]),
    _fwd('small_c1_55s2', 65537, 5, 9, 1, 1, 5, 2, 2, pv=0.5, kernels=[small_fwd(5, 5, 2, 2, 1, 1, 8)]),
    _fwd('small_c1_55s2_4', 65537, 3, 5, 1, 4, 5, 2, 2, kernels=[small_fwd(5, 5, 2, 2, 1, 4, 4)]),
    _fwd('small_c1_53_64', 65537, 5, 4, 1, 64, (5, 3), (0, 1), (2, 1), kernels=[small_fwd(5, 3, 2, 1, 1, 16, 4)]),
    # Cin > 1
    _fwd('small_16_1', 2, 19, 37, 16, 1, 3, 1, kernels=[small_fwd(3, 3, 1, 1, 16, 1, 8)]),
    _fwd('small_16_1_ups', 2, 20, 38, 16, 1, 3, 1, pv=0.5, ups=2, kernels=[small_fwd(3, 3, 1, 1, 16, 1, 8, 2)]),
    _fwd('small_44_s2', 2, 21, 43, 4, 4, 5, 2, 2, pv=0.5, kernels=[small_fwd(5, 5, 2, 2, 4, 4, 4)]),
    _fwd('small_44_s1', 2, 19, 37, 4, 4, 5, 2, kernels=[small_fwd(5, 5, 1, 1, 4, 4, 4)]),
    _fwd('small_44_s1_ups', 2, 20, 38, 4, 4, 5, 2, pv=0.5, ups=2, kernels=[small_fwd(5, 5, 1, 1, 4, 4, 4, 2)]),
    _fwd('small_42', 2, 19, 37, 4, 2, 5, 2, kernels=[small_fwd(5, 5, 1, 1, 4, 2, 4)]),
    _fwd('small_42_ups', 2, 20, 38, 4, 2, 5, 2, pv=0.5, ups=2, kernels=[small_fwd(5, 5, 1, 1, 4, 2, 4, 2)]),
    _fwd('small_24', 2, 19, 37, 2, 4, 5, 2, kernels=[small_fwd(5, 5, 1, 1, 2, 4, 4)]),
    _fwd('small_24_ups', 2, 20, 38, 2, 4, 5, 2, pv=-1.0, ups=2, kernels=[small_fwd(5, 5, 1, 1, 2, 4, 4, 2)]),
    # the general kernel: Cin = 3 has no fast kernel
    _fwd('direct_48', 2, 13, 17, 3, 48, 3, 1, pv=0.5, kernels=[fwd_direct(48)]),
    _fwd('direct_24', 2, 13, 17, 3, 24, 3, 2, 2, kernels=[fwd_direct(24)]),
    _fwd('direct_12', 2, 13, 17, 3, 12, (5, 3), (2, 1), (2, 1), pv=-1.0, kernels=[fwd_direct(12)]),
    _fwd('direct_6', 2, 13, 17, 3, 6, 3, 0, kernels=[fwd_direct(6)]),
    _fwd('direct_5', 2, 14, 18, 3, 5, 3, 1, ups=2, kernels=[fwd_direct(5)]),

    # ---------------------------------------------------------------- input gradient, FP32 mode (conv_bwd_fast.cu)
    # stride 1: the forward stencils on flipped weights (padding kh - 1 - ph)
    *[_dgrad(f'flip_55_11_p{p}', 2, 37, 132 if p == 2 else 70, 1, 1, 5, p,
             kernels=[FLIP, 'conv55_c1_tile_kernel' if p == 2 else c1_fwd(5, 5, 1, 1, 1)]) for p in range(5)],
    *[_dgrad(f'flip_33_1_16_p{p}', 2, 19, 37, 1, 16, 3, p, kernels=[FLIP, small_fwd(3, 3, 1, 1, 16, 1, 8)])
      for p in range(3)],
    *[_dgrad(f'flip_33_16_1_p{p}', 2, 35, 70, 16, 1, 3, p, kernels=[FLIP, c1_fwd(3, 3, 1, 1, 16)]) for p in range(3)],
    *[_dgrad(f'flip_55_44_p{p}', 2, 19, 37, 4, 4, 5, (p, 4 - p), kernels=[FLIP, small_fwd(5, 5, 1, 1, 4, 4, 4)])
      for p in range(5)],
    *[_dgrad(f'flip_55_42_p{p}', 2, 19, 37, 4, 2, 5, p, kernels=[FLIP, small_fwd(5, 5, 1, 1, 2, 4, 4)])
      for p in range(5)],
    *[_dgrad(f'flip_55_24_p{p}', 2, 19, 37, 2, 4, 5, p, kernels=[FLIP, small_fwd(5, 5, 1, 1, 4, 2, 4)])
      for p in range(5)],
    _dgrad('gather_55_11_p5', 2, 13, 21, 1, 1, 5, 5, kernels=[dgrad_direct(1)]),
    # strided, COUT <= 4
    *[_dgrad(f'small_dgrad_{ci}{co}_ph{ph}', 2, 37, 43, ci, co, 5, (ph, 2), 2,
             kernels=[f'conv_small_dgrad_kernel<5,5,2,2,2,{ci},{co},{8 if ci == 1 else 4}>'])
      for ci, co in ((1, 1), (1, 4), (4, 4)) for ph in (0, 2, 3)],
    # Cin = 1, 5x3: output-side scatter with float atomics (exact on integers)
    *[_dgrad(f'scatter_{co}_s{s[0]}{s[1]}_ph{ph}', 2, 23, 41, 1, co, (5, 3), (ph, 1), s,
             kernels=['conv_dgrad_cin1_scatter_kernel<5,3>'])
      for co in (4, 64, 256) for s in ((2, 1), (2, 2), (1, 2)) for ph in (0, 2)],
    # Cin = 1, Cout % 64 == 0: warp per input pixel
    _dgrad('warp_55s2_64', 2, 23, 41, 1, 64, 5, 2, 2, kernels=['conv_dgrad_cin1_warp_kernel']),
    _dgrad('warp_33s2_128', 2, 23, 41, 1, 128, 3, 1, 2, kernels=['conv_dgrad_cin1_warp_kernel']),
    _dgrad('warp_99s1_64', 1, 21, 30, 1, 64, 9, 4, kernels=['conv_dgrad_cin1_warp_kernel']),
    # the general gather kernel
    *[_dgrad(f'dgrad_direct_{ci}', 2, 15, 19, ci, 3, 3, 1, 2, kernels=[dgrad_direct(ci)]) for ci in (8, 4, 2, 1)],

    # ---------------------------------------------------------------- weight gradient, FP32 mode
    _wgrad('tiled_4', 1, 20, 70, 4, 4, 5, 2, kernels=['conv55_c4_wgrad_tiled_kernel<4,false>', FINALIZE]),
    _wgrad('tiled_2', 2, 17, 66, 4, 2, 5, 2, kernels=['conv55_c4_wgrad_tiled_kernel<2,false>', FINALIZE]),
    _wgrad('tiled_4_ups', 1, 20, 70, 4, 4, 5, 2, ups=2, kernels=['conv55_c4_wgrad_tiled_kernel<4,true>', FINALIZE]),
    _wgrad('tiled_2_ups', 2, 18, 66, 4, 2, 5, 2, ups=2, kernels=['conv55_c4_wgrad_tiled_kernel<2,true>', FINALIZE]),
    # 12 x 9 x 5 = 540 tiles on the 444-CTA persistent grid
    _wgrad('tiled_4_540', 12, 130, 260, 4, 4, 5, 2, kernels=['conv55_c4_wgrad_tiled_kernel<4,false>', FINALIZE]),
    _wgrad('tiled_2_ups_540', 12, 130, 260, 4, 2, 5, 2, ups=2,
           kernels=['conv55_c4_wgrad_tiled_kernel<2,true>', FINALIZE]),
    _wgrad('roll', 2, 37, 40, 1, 1, 5, 2, kernels=['conv55_c1_wgrad_roll_kernel<16,false>', FINALIZE]),
    _wgrad('roll_pv', 1, 53, 72, 1, 1, 5, 2, pv=0.5, kernels=['conv55_c1_wgrad_roll_kernel<16,false>', FINALIZE]),
    _wgrad('roll_ups', 2, 38, 40, 1, 1, 5, 2, ups=2, kernels=['conv55_c1_wgrad_roll_kernel<16,true>', FINALIZE]),
    _wgrad('roll_ups_pv', 1, 54, 72, 1, 1, 5, 2, pv=-1.0, ups=2,
           kernels=['conv55_c1_wgrad_roll_kernel<16,true>', FINALIZE]),
    _wgrad('small_33_1_16', 2, 37, 38, 1, 16, 3, 1, pv=0.5, kernels=[small_wgrad(3, 3, 1, 1, 1, 1, 4, 4, 16), FINALIZE]),
    _wgrad('small_33_16_1', 2, 37, 38, 16, 1, 3, 1, kernels=[small_wgrad(3, 3, 1, 1, 16, 4, 1, 4, 16), FINALIZE]),
    _wgrad('small_33_4_1', 2, 35, 43, 4, 1, 3, 0, pv=-1.0, kernels=[small_wgrad(3, 3, 1, 1, 4, 4, 1, 4, 16), FINALIZE]),
    _wgrad('small_55s1_11', 2, 37, 37, 1, 1, 5, 2, kernels=[small_wgrad(5, 5, 1, 1, 1, 1, 1, 8, 16), FINALIZE]),
    _wgrad('small_55s2_11', 2, 37, 43, 1, 1, 5, 2, 2, pv=0.5, kernels=[small_wgrad(5, 5, 2, 2, 1, 1, 1, 4, 4), FINALIZE]),
    _wgrad('small_55s2_14', 2, 37, 43, 1, 4, 5, 2, 2, kernels=[small_wgrad(5, 5, 2, 2, 1, 1, 2, 4, 2), FINALIZE]),
    _wgrad('small_55s2_44', 2, 37, 43, 4, 4, 5, 2, 2, kernels=[small_wgrad(5, 5, 2, 2, 4, 4, 1, 4, 2), FINALIZE]),
    _wgrad('small_55s1_44_pv', 2, 21, 38, 4, 4, 5, 2, pv=0.5, kernels=[small_wgrad(5, 5, 1, 1, 4, 4, 1, 4, 8), FINALIZE]),
    _wgrad('small_55s1_44_p1', 2, 21, 39, 4, 4, 5, 1, kernels=[small_wgrad(5, 5, 1, 1, 4, 4, 1, 4, 8), FINALIZE]),
    _wgrad('small_53_1_16', 2, 41, 37, 1, 16, (5, 3), (0, 1), (2, 1),
           kernels=[small_wgrad(5, 3, 2, 1, 1, 1, 4, 4, 7), FINALIZE]),
    _wgrad('tile_64_64', 2, 30, 41, 3, 40, 3, 1, pv=0.5, kernels=[wgrad_tile(40), 'conv_wgrad_reduce_kernel']),
    _wgrad('tile_64_16', 2, 30, 41, 3, 12, 3, 1, 2, kernels=[wgrad_tile(12), 'conv_wgrad_reduce_kernel']),
    _wgrad('tile_32_8', 3, 30, 41, 3, 5, (5, 3), (2, 1), (2, 1), pv=-1.0,
           kernels=[wgrad_tile(5), 'conv_wgrad_reduce_kernel']),
    # in_upsample = 2 where no weight-gradient kernel reads the half-resolution input: an error, dw / db untouched
    _wgrad('ups_none_11_wo38', 1, 20, 38, 1, 1, 5, 2, ups=2, kernels=None),
    _wgrad('ups_none_44_pv', 1, 20, 40, 4, 4, 5, 2, pv=0.5, ups=2, kernels=None),
    _wgrad('ups_none_33_1_16', 1, 20, 40, 1, 16, 3, 1, ups=2, kernels=None),
    _wgrad('ups_none_33_16_1', 1, 20, 40, 16, 1, 3, 1, ups=2, kernels=None),

    # ---------------------------------------------------------------- TF32 mode (tc_gemm.cu, conv_row_tc.cu)
    *[r for name, (n, h, w), cin, cout, k, p, s in (
        ('char2', (3, 14, 256), 64, 64, (5, 3), (0, 1), (2, 1)),
        ('char2_b64', (64, 14, 256), 64, 64, (5, 3), (0, 1), (2, 1)),
        ('ragged', (2, 14, 70), 64, 64, (5, 3), (0, 1), (2, 1)),
        ('c32_48', (2, 9, 131), 32, 48, 3, 1, 1),
        ('c32_64', (2, 11, 67), 32, 64, 3, 1, 1),
        ('c128_32', (1, 9, 40), 128, 32, (2, 3), 1, (2, 1)))
      for r in (
        _fwd(f'tc_fwd_{name}', n, h, w, cin, cout, k, p, s, mode=TF32, kernels=['tc_conv_slab_kernel']),
        _dgrad(f'tc_dgrad_{name}', n, h, w, cin, cout, k, p, s, mode=TF32,
               kernels=['tc_gemm_kernel<2>' if cout % 32 == 0 else dgrad_direct(cin)]),
        _wgrad(f'tc_wgrad_{name}', n, h, w, cin, cout, k, p, s, mode=TF32,
               kernels=['tc_gemm_kernel<4>' if cout % 32 == 0 else wgrad_tile(cout)]))],
    # an output the slab kernel cannot store with 16-byte stores: the one-tile-per-CTA implicit GEMM
    _fwd('tc_fwd_gemm_char2', 3, 14, 256, 64, 64, (5, 3), (0, 1), (2, 1), mode=TF32, shift=('y',),
         kernels=['tc_gemm_kernel<1>']),
    _fwd('tc_fwd_gemm_c32_48', 2, 9, 131, 32, 48, 3, 1, mode=TF32, shift=('y',), kernels=['tc_gemm_kernel<1>']),
    _fwd('row_tc_44', 2, 37, 70, 4, 4, 5, 2, mode=TF32, kernels=['conv55_row_tc_kernel<4,false>']),
    _fwd('row_tc_42', 2, 37, 70, 4, 2, 5, 2, mode=TF32, kernels=['conv55_row_tc_kernel<2,false>']),
    _fwd('row_tc_44_ups', 2, 38, 70, 4, 4, 5, 2, ups=2, mode=TF32, kernels=['conv55_row_tc_kernel<4,true>']),
    _fwd('row_tc_42_ups', 1, 30, 70, 4, 2, 5, 2, ups=2, mode=TF32, kernels=['conv55_row_tc_kernel<2,true>']),
    _dgrad('row_tc_dgrad_44', 2, 37, 70, 4, 4, 5, 2, mode=TF32, kernels=[FLIP, 'conv55_row_tc_kernel<4,false>']),
    _dgrad('row_tc_dgrad_24', 2, 37, 70, 2, 4, 5, 2, mode=TF32, kernels=[FLIP, 'conv55_row_tc_kernel<2,false>']),
]

_BY_ID = {r.id: r for r in ROWS}


def _fallback(row_id):
    """The row on unaligned views, with the general kernel that must run instead (None: the call must fail)."""
    r = _BY_ID[row_id]
    if r.op == 'fwd':
        k = fwd_direct(r.cout)
    elif r.op == 'wgrad':
        k = wgrad_tile(r.cout) if r.ups == 1 else None      # the general kernel reads no half-resolution input
    elif r.sh == 1 and r.sw == 1 and r.kh - 1 - r.ph >= 0 and r.kw - 1 - r.pw >= 0 and \
            r.kh * r.kw * r.cin * r.cout <= 4096:
        k = fwd_direct(r.cin)                   # stride-1 dgrad: flipped weights, then the general forward kernel
    else:
        k = dgrad_direct(r.cin)
    return r.unaligned(k)


ROWS += [_fallback(i) for i in (
    'c55_tile', 'c55_ups_tile', 'c1_55s1_w70', 'c1_55s2_4', 'c1_33_16_p1', 'c1_53_16_ph0', 'wide64', 'small_16_1_ups',
    'small_44_s2', 'small_44_s1', 'small_42', 'small_24', 'flip_55_11_p2', 'flip_33_1_16_p1', 'flip_55_44_p1',
    'small_dgrad_11_ph2', 'small_dgrad_14_ph3', 'small_dgrad_44_ph0', 'scatter_64_s21_ph0', 'warp_55s2_64', 'tiled_4',
    'tiled_2_ups', 'roll_pv', 'roll_ups', 'small_33_1_16', 'small_33_16_1', 'small_33_4_1', 'small_55s1_11',
    'small_55s2_11', 'small_55s2_14', 'small_55s2_44', 'small_55s1_44_pv', 'small_53_1_16', 'tc_fwd_char2',
    'tc_dgrad_char2', 'tc_wgrad_c32_64', 'row_tc_44_ups', 'row_tc_dgrad_44')]
_BY_ID = {r.id: r for r in ROWS}
assert len(_BY_ID) == len(ROWS), 'duplicate row id'

# epilogue / accumulation variants run by each row: (bias flag, activation) and (accumulate, bias flag)
FWD_VARIANTS = ((1, NONE), (0, LEAKY), (1, LEAKY), (1, SIGMOID))
WGRAD_VARIANTS = ((0, 1), (1, 1), (0, 0), (1, 0))


# ------------------------------------------------------------------------------------------------ helpers
def _rng(row_id):
    return np.random.default_rng(zlib.crc32(row_id.encode()))


def _ints(rng, lo, hi, shape):
    return rng.integers(lo, hi + 1, size=shape).astype(np.float64)


def _upload(nn, a, shifted):
    """float32 device copy of `a`; shifted: a view that starts one float past a 16-byte aligned block."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    if not shifted:
        return nn.CP.copy(a)
    d = nn.CP.copy(np.concatenate([np.zeros(1, np.float32), a.ravel()]))
    return d.flat_view(1, a.size, a.shape)


def _filled(nn, shape, value, shifted):
    size = int(np.prod(shape))
    d = nn.DeviceArray.full((size + (1 if shifted else 0),), value)
    return d.flat_view(1 if shifted else 0, size, shape)


def _host(d):
    return np.asarray(d.get(), dtype=np.float64)


def _act(v, act):
    if act == LEAKY:
        return O.leaky_relu_fwd(v, ALPHA)
    if act == SIGMOID:
        return O.sigmoid_fwd(v)
    return v


def rna_tf32(v):
    """float32 -> TF32 rounded to nearest, ties away from zero (cvt.rna.tf32.f32)."""
    u = np.asarray(v, dtype=np.float32).view(np.uint32)
    return ((u + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32).astype(np.float64)


def trunc_tf32(v):
    """float32 -> TF32 by truncation, as the tensor core reads an FP32 operand."""
    u = np.asarray(v, dtype=np.float32).view(np.uint32)
    return (u & np.uint32(0xFFFFE000)).view(np.float32).astype(np.float64)


def tc_scaled(w):
    """The operand the TMEM-window kernels (conv_row_tc.cu, conv_pair_tc.cu, conv_pair_rows_tc.cu) multiply by: they
    read their other operand truncated to TF32 and make that unbiased by scaling these weights by (1 + 2^-11) before
    rounding them to TF32.  On integers the truncation loses nothing, so the scaling shows: each |w| in {1, 2} becomes
    |w| (1 + 2^-10).  The kernels are exact with respect to these operands, not to w."""
    return rna_tf32(np.float32(w) * np.float32(1.0 + 2.0 ** -11))


def assert_exact(got, want, what):
    assert got.shape == want.shape, f'{what}: shape {got.shape} != {want.shape}'
    bad = got != want
    if bad.any():
        idx = tuple(int(i[0]) for i in np.nonzero(bad))
        pytest.fail(f'{what}: {int(bad.sum())} of {bad.size} elements differ from the exact oracle; first at {idx}: '
                    f'got {got[idx]!r}, want {want[idx]!r}')


def assert_sigmoid(got, want, what):
    assert got.shape == want.shape, f'{what}: shape {got.shape} != {want.shape}'
    np.testing.assert_allclose(got, want, rtol=1e-4, atol=2e-6 * max(float(np.abs(want).max()), 1e-30), err_msg=what)


def assert_exact_regime(*bounds):
    """Each argument: the oracle on |operands| -- an upper bound of every partial sum the kernels form."""
    for b in bounds:
        m = float(np.max(np.abs(b))) if np.size(b) else 0.0
        assert m <= EXACT_LIMIT, f'row leaves the exact regime: a partial sum may reach {m:.0f} > 2^22'


class _Operands:
    def __init__(self, row):
        rng = _rng(row.id)
        self.x = _ints(rng, -2, 2, (row.n, row.h // row.ups, row.w // row.ups, row.cin))
        self.w = _ints(rng, -2, 2, (row.kh, row.kw, row.cin, row.cout))
        self.b = _ints(rng, -4, 4, (row.cout,))
        self.dy = _ints(rng, -2, 2, (row.n, row.ho, row.wo, row.cout))
        self.dw0 = _ints(rng, -4, 4, self.w.shape)
        self.db0 = _ints(rng, -4, 4, self.b.shape)

    def x_logical(self, row, x=None):
        x = self.x if x is None else x
        return O.upsample2d_fwd(x, 2) if row.ups == 2 else x


def _conv_args(row):
    return dict(padding=(row.ph, row.pw), stride=(row.sh, row.sw))


class _Call:
    """Device operands of one row and the library call for one variant."""

    def __init__(self, nn, row, ops):
        self.nn, self.row = nn, row
        sh = row.shift
        self.x = _upload(nn, ops.x, 'x' in sh)
        self.w = _upload(nn, ops.w, 'w' in sh)
        self.b = _upload(nn, ops.b, 'b' in sh)
        self.dy = _upload(nn, ops.dy, 'dy' in sh)
        self.ops = ops
        if row.op == 'wgrad':
            need = ctypes.c_size_t(0)
            from univer_ocr_b200._lib import lib
            lib.uocr_conv2d_wgrad_workspace(ctypes.byref(row.desc()), ctypes.byref(need))
            self.ws_bytes = need.value
            self.ws = nn.DeviceArray((max(need.value, 4) + 3) // 4)

    def launch(self, variant, grads=None):
        from univer_ocr_b200._lib import lib
        nn, row = self.nn, self.row
        d = row.desc()
        st = nn.CP.stream()
        if row.op == 'fwd':
            d.bias, act = variant
            out = _filled(nn, (row.n, row.ho, row.wo, row.cout), float('nan'), 'y' in row.shift)
            lib.uocr_conv2d_fwd(ctypes.byref(d), self.x.ptr, self.w.ptr, self.b.ptr, out.ptr, act, ALPHA, st)
            return out
        if row.op == 'dgrad':
            out = _filled(nn, (row.n, row.h, row.w, row.cin), float('nan'), 'dx' in row.shift)
            lib.uocr_conv2d_dgrad(ctypes.byref(d), self.dy.ptr, self.w.ptr, out.ptr, st)
            return out
        acc, d.bias = variant
        dw, db = grads or (_upload(nn, self.ops.dw0, 'w' in row.shift), _upload(nn, self.ops.db0, 'b' in row.shift))
        lib.uocr_conv2d_wgrad(ctypes.byref(d), self.x.ptr, self.dy.ptr, dw.ptr, db.ptr, acc, self.ws.ptr,
                              self.ws_bytes, st)
        return dw, db


def check_row(nn, row):
    from univer_ocr_b200._lib import UocrError
    ops = _Operands(row)
    call = _Call(nn, row, ops)
    xl, kw = ops.x_logical(row), _conv_args(row)
    xa, wa, dya = np.abs(xl), np.abs(ops.w), np.abs(ops.dy)
    w = ops.w
    if any('conv55_row_tc_kernel' in k for k in row.kernels or ()):
        w = tc_scaled(ops.w)
    if row.op == 'fwd':
        assert_exact_regime(O.conv2d_fwd(xa, wa, np.abs(ops.b), padding_value=abs(row.pv), **kw))
        y0 = O.conv2d_fwd(xl, w, ops.b, padding_value=row.pv, bias=False, **kw)
        for bias, act in FWD_VARIANTS:
            want = _act(y0 + bias * ops.b, act)
            got = _host(call.launch((bias, act)))
            what = f'{row.id} fwd bias={bias} act={act}'
            (assert_sigmoid if act == SIGMOID else assert_exact)(got, want, what)
        return
    if row.op == 'dgrad':
        assert_exact_regime(O.conv2d_bwd(xa, wa, dya, **kw)[0])
        want = O.conv2d_bwd(xl, w, ops.dy, padding_value=row.pv, **kw)[0]
        assert_exact(_host(call.launch(None)), want, f'{row.id} dgrad')
        return
    _, gw_abs, gb_abs = O.conv2d_bwd(xa, wa, dya, padding_value=abs(row.pv), **kw)
    assert_exact_regime(gw_abs + np.abs(ops.dw0), gb_abs + np.abs(ops.db0))
    _, gw, gb = O.conv2d_bwd(xl, ops.w, ops.dy, padding_value=row.pv, **kw)
    for acc, bias in WGRAD_VARIANTS:
        what = f'{row.id} wgrad accumulate={acc} bias={bias}'
        if row.kernels is None:
            dw, db = _upload(nn, ops.dw0, False), _upload(nn, ops.db0, False)
            with pytest.raises(UocrError, match='in_upsample'):
                call.launch((acc, bias), (dw, db))
            assert_exact(_host(dw), ops.dw0, what + ' dw untouched')
            assert_exact(_host(db), ops.db0, what + ' db untouched')
            continue
        dw, db = call.launch((acc, bias))
        assert_exact(_host(dw), gw + acc * ops.dw0, what + ' dw')
        assert_exact(_host(db), bias * gb + acc * ops.db0, what + ' db')


@pytest.mark.parametrize('row_id', [r.id for r in ROWS])
def test_conv_kernel_exact(nn, row_id):
    check_row(nn, _BY_ID[row_id])


# ------------------------------------------------------------------------------------------------ pair kernels
# the shapes of test_monochrome_pair_on_tensor_cores: the TF32 row kernel (W % 4 == 0, W >= 8) and the TMEM kernel
PAIR_FWD_SHAPES = [(2, 16, 256), (3, 21, 150), (1, 5, 3), (2, 1, 1), (1, 63, 31), (1, 130, 61), (5, 3, 240),
                   (2, 496, 736), (3, 33, 244), (2, 40, 248), (1, 7, 492), (1, 130, 1000), (5, 3, 12), (1, 2, 8),
                   (9, 300, 736), (9, 300, 734)]
# ragged 16-row groups and 8-column strips
PAIR_BWD_SHAPES = [(2, 16, 256), (3, 21, 150), (1, 5, 3), (2, 1, 1), (1, 130, 61), (2, 37, 45), (1, 33, 250)]


def _pair_operands(key):
    rng = _rng(key)
    n, h, w = key_shape = tuple(int(v) for v in key.split('_')[-1].split('x'))
    x = _ints(rng, -2, 2, (n, h, w, 1))
    w1 = _ints(rng, -2, 2, (3, 3, 1, 16))
    b1 = _ints(rng, -4, 4, (16,))
    w2 = _ints(rng, -2, 2, (3, 3, 16, 1))
    b2 = _ints(rng, -4, 4, (1,))
    dy = _ints(rng, -2, 2, (n, h, w, 1))
    return key_shape, x, w1, b1, w2, b2, dy


def _pair_kernel_fwd(shape, c_mid, act1, mode):
    leaky = 'true' if act1 == LEAKY else 'false'
    if mode == TF32 and c_mid == 16:
        if shape[2] % 4 == 0 and shape[2] >= 8:
            return f'conv3x3_pair_rows_kernel<{leaky},false>'
        return f'conv3x3_pair_tmem_kernel<{leaky},false>'
    return f'conv3x3_pair_fwd_kernel<8,16,{leaky}>'


def _shape_id(shape):
    return 'x'.join(str(v) for v in shape)


def _pair_fwd_launch(nn, d, shape, c_mid, act1, mode):
    from univer_ocr_b200._lib import lib
    n, h, w = shape
    y = _filled(nn, (n, h, w, 1), float('nan'), False)
    lib.uocr_conv3x3_pair_fwd(d['x'].ptr, d['w1_%d' % c_mid].ptr, d['b1_%d' % c_mid].ptr, d['w2_%d' % c_mid].ptr,
                              d['b2'].ptr, y.ptr, n, h, w, c_mid, act1, ALPHA, NONE, 0.0, mode, nn.CP.stream())
    return y


def _pair_device(nn, x, w1, b1, w2, b2, dy):
    d = {'x': _upload(nn, x, False), 'b2': _upload(nn, b2, False), 'dy': _upload(nn, dy, False)}
    for c in (16, 5):
        d['w1_%d' % c] = _upload(nn, w1[..., :c], False)
        d['b1_%d' % c] = _upload(nn, b1[:c], False)
        d['w2_%d' % c] = _upload(nn, w2[:, :, :c, :], False)
    return d


@pytest.mark.parametrize('shape', PAIR_FWD_SHAPES, ids=_shape_id)
def test_pair_fwd_exact(nn, shape):
    """uocr_conv3x3_pair_fwd in FP32 (CUDA-core kernel) and TF32 mode (row / TMEM tensor-core kernels for c_mid 16,
    the CUDA-core kernel for c_mid 5), act1 LeakyRelu 0.25 or none, act2 none: bit-exact against the oracle chain."""
    _, x, w1, b1, w2, b2, _ = _pair_operands('pair_fwd_' + _shape_id(shape))
    xa = np.abs(x)
    assert_exact_regime(O.conv2d_fwd(O.conv2d_fwd(xa, np.abs(w1), np.abs(b1), 1), np.abs(w2), np.abs(b2), 1))
    d = _pair_device(nn, x, w1, b1, w2, b2, x)
    for c in (16, 5):
        pre = O.conv2d_fwd(x, w1[..., :c], b1[:c], 1)
        # the tensor-core kernels (c_mid 16): w1, b1 scaled as tc_scaled says, the hidden map read truncated to TF32
        pre_tc = O.conv2d_fwd(x, tc_scaled(w1[..., :c]), tc_scaled(b1[:c]), 1)
        for act1 in (LEAKY, NONE):
            want = O.conv2d_fwd(_act(pre, act1), w2[:, :, :c, :], b2, 1)
            want_tc = O.conv2d_fwd(trunc_tf32(_act(pre_tc, act1)), w2[:, :, :c, :], b2, 1)
            for mode in (FP32, TF32):
                got = _host(_pair_fwd_launch(nn, d, shape, c, act1, mode))
                tc = mode == TF32 and c == 16
                assert_exact(got, want_tc if tc else want, f'pair fwd {shape} c_mid={c} act1={act1} mode={mode}')


def _pair_bwd_launch(nn, d, shape, act1, mode, with_dx, acc, init):
    from univer_ocr_b200._lib import lib
    n, h, w = shape
    need = ctypes.c_size_t(0)
    lib.uocr_conv3x3_pair_bwd_workspace(n, h, w, 16, ctypes.byref(need))
    ws = nn.DeviceArray(((need.value + 3) // 4,))
    g = [_upload(nn, a, False) for a in init]
    dx = _filled(nn, (n, h, w, 1), float('nan'), False) if with_dx else None
    args = (d['x'].ptr, d['w1_16'].ptr, d['b1_16'].ptr, d['w2_16'].ptr, d['dy'].ptr, dx.ptr if with_dx else None,
            g[0].ptr, g[1].ptr, g[2].ptr, g[3].ptr, n, h, w, 16, act1, ALPHA, acc, ws.ptr, need.value)
    if mode is None:
        lib.uocr_conv3x3_pair_bwd(*args, nn.CP.stream())
    else:
        lib.uocr_conv3x3_pair_bwd_mode(*args, mode, nn.CP.stream())
    return g, dx


def _pair_bwd_kernels(act1, mode, with_dx):
    if mode == TF32:
        k = ['conv3x3_pair_wgrad_tc_kernel<%s,false>' % ('true' if act1 == LEAKY else 'false')]
    else:
        k = ['conv3x3_pair_wgrad_kernel<8,16>']
    k.append('conv3x3_pair_wgrad_finalize_kernel')
    if with_dx:
        k.append('conv3x3_pair_dgrad_kernel<8,16>')
    return k


@pytest.mark.parametrize('shape', PAIR_BWD_SHAPES, ids=_shape_id)
def test_pair_bwd_exact(nn, shape):
    """uocr_conv3x3_pair_bwd (FP32 CUDA-core kernels) and uocr_conv3x3_pair_bwd_mode in TF32 mode (tensor-core weight
    gradients), with and without dx, overwriting and accumulating: bit-exact against the oracle's layer-by-layer
    backward of conv -> LeakyRelu 0.25 (or none) -> conv."""
    _, x, w1, b1, w2, b2, dy = _pair_operands('pair_bwd_' + _shape_id(shape))
    rng = _rng('pair_bwd_init_' + _shape_id(shape))
    init = [_ints(rng, -4, 4, s) for s in ((3, 3, 1, 16), (16,), (3, 3, 16, 1), (1,))]
    xa, w1a, b1a, w2a, dya = np.abs(x), np.abs(w1), np.abs(b1), np.abs(w2), np.abs(dy)
    ha = O.conv2d_fwd(xa, w1a, b1a, 1)
    dha, dw2a, db2a = O.conv2d_bwd(ha, w2a, dya, 1)
    dxa, dw1a, db1a = O.conv2d_bwd(xa, w1a, dha, 1)
    assert_exact_regime(ha, dha, dxa, dw1a + 4, db1a + 4, dw2a + 4, db2a + 4)
    d = _pair_device(nn, x, w1, b1, w2, b2, dy)
    pre = O.conv2d_fwd(x, w1, b1, 1)
    for act1 in (LEAKY, NONE):
        dact, odw2, odb2 = O.conv2d_bwd(_act(pre, act1), w2, dy, 1)
        dpre = O.leaky_relu_bwd(pre, dact, ALPHA) if act1 == LEAKY else dact
        odx, odw1, odb1 = O.conv2d_bwd(x, w1, dpre, 1)
        for mode in (None, FP32, TF32):
            for with_dx, acc in ((True, 0), (False, 1), (True, 1)):
                g, dx = _pair_bwd_launch(nn, d, shape, act1, mode, with_dx, acc, init)
                what = f'pair bwd {shape} act1={act1} mode={mode} dx={with_dx} accumulate={acc}'
                for name, got, want, i0 in zip(('dw1', 'db1', 'dw2', 'db2'), g, (odw1, odb1, odw2, odb2), init):
                    assert_exact(_host(got), want.reshape(i0.shape) + acc * i0, f'{what} {name}')
                if with_dx:
                    assert_exact(_host(dx), odx, f'{what} dx')


# ------------------------------------------------------------------------------------------------ kernel reach
def _reach_cases():
    cases = [pytest.param(('conv', r.id), r.kernels, id=r.id) for r in ROWS if r.kernels is not None]
    for shape in PAIR_FWD_SHAPES[:3] + [PAIR_FWD_SHAPES[4]]:
        for c, act1, mode in ((16, LEAKY, FP32), (16, NONE, FP32), (16, LEAKY, TF32), (16, NONE, TF32),
                              (5, LEAKY, TF32)):
            cases.append(pytest.param(('pair_fwd', shape, c, act1, mode), [_pair_kernel_fwd(shape, c, act1, mode)],
                                      id=f'pair_fwd_{_shape_id(shape)}_c{c}_act{act1}_mode{mode}'))
    for act1, mode, with_dx in ((LEAKY, None, True), (LEAKY, TF32, False), (NONE, TF32, True)):
        cases.append(pytest.param(('pair_bwd', (2, 37, 45), act1, mode, with_dx), _pair_bwd_kernels(act1, mode, with_dx),
                                  id=f'pair_bwd_act{act1}_mode{mode}_dx{int(with_dx)}'))
    return cases


def _launch_case(nn, case):
    if case[0] == 'conv':
        row = _BY_ID[case[1]]
        call = _Call(nn, row, _Operands(row))
        call.launch(FWD_VARIANTS[0] if row.op == 'fwd' else WGRAD_VARIANTS[0] if row.op == 'wgrad' else None)
        return
    shape = case[1]
    _, x, w1, b1, w2, b2, dy = _pair_operands('pair_reach_' + _shape_id(shape))
    d = _pair_device(nn, x, w1, b1, w2, b2, dy)
    if case[0] == 'pair_fwd':
        _pair_fwd_launch(nn, d, shape, *case[2:])
    else:
        init = [np.zeros(s) for s in ((3, 3, 1, 16), (16,), (3, 3, 16, 1), (1,))]
        _pair_bwd_launch(nn, d, shape, case[2], case[3], case[4], 0, init)


@pytest.mark.parametrize('case,kernels', _reach_cases())
def test_each_row_reaches_its_kernel(nn, case, kernels):
    """The exact comparisons only say something about the kernel that actually ran: record the CUDA kernels of the
    row's call with torch.profiler and require the row's kernel instantiations among them (demangled names, whitespace
    removed)."""
    torch = pytest.importorskip('torch')
    from torch.profiler import ProfilerActivity, profile
    if not torch.cuda.is_available():
        pytest.skip('torch sees no CUDA device')
    torch.cuda.init()
    _launch_case(nn, case)                      # warm-up outside the trace: module loading, pool growth
    nn.CP.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _launch_case(nn, case)
        nn.CP.synchronize()
    names = [''.join(e.name.split()) for e in prof.events() if 'kernel' in e.name or '<' in e.name]
    if not names:
        pytest.skip('torch.profiler recorded no kernel launched by libuocr.so in this process')
    for k in kernels:
        k = ''.join(k.split())
        assert any(k + '(' in n or n.endswith(k) for n in names), f'{k} did not run; launched: {sorted(set(names))}'
