"""CPU: tfcb_gdn_native_16bit, the library's answer to "does this 16-bit GDN call run natively?", over a grid of
configurations, against the predicate functional.py evaluated itself before it asked the library (kept here as the
reference).  The query reads no memory and touches no device, so fake addresses stand in for tensors."""
import itertools

import pytest

from compression_b200 import _lib
from compression_b200.functional import GDN_INVERSE, GDN_POW_ALPHA, GDN_POW_EPSILON, GDN_RECTIFY

ALIGNED, MISALIGNED = 1 << 20, (1 << 20) + 2  # the second is one 16-bit element past a 16-byte boundary


def _former_python_predicate(dtype, C, n_pix, alpha, epsilon, pow_alpha, pow_epsilon, x, beta, dy=None, boxes=True):
  """functional._native16 on addresses instead of tensors (the caller checked that dy has x's type).  The forward
  passed boxes = C != 128 and no dy, the backward dy and boxes = True."""
  return (dtype in (1, 2) and C in (128, 192) and not pow_alpha and not pow_epsilon and
          float(alpha) in (1.0, 2.0) and float(epsilon) in (1.0, 0.5) and n_pix > 0 and
          (n_pix < 2**31 or not boxes) and
          all(p % 16 == 0 for p in (x, beta) + (() if dy is None else (dy,))))


@pytest.mark.parametrize("backward", [False, True])
@pytest.mark.parametrize("C", [64, 128, 192])
def test_native_16bit_query_keeps_the_former_python_predicate(backward, C):
  lib = _lib.lib()
  grid = itertools.product((0, 1, 2, 3), (1.0, 2.0, 3.0), (1.0, 0.5, 2.0), (False, True), (False, True),
                           (0, GDN_INVERSE | GDN_RECTIFY), (0, 1, 2**31 - 1, 2**31),
                           (ALIGNED, MISALIGNED), (ALIGNED, MISALIGNED), (ALIGNED, MISALIGNED))
  checked = 0
  for dtype, alpha, epsilon, pow_alpha, pow_epsilon, flags, n_pix, x, beta, dy in grid:
    flags |= (GDN_POW_ALPHA if pow_alpha else 0) | (GDN_POW_EPSILON if pow_epsilon else 0)
    got = lib.tfcb_gdn_native_16bit(int(backward), x, beta, dy, n_pix, C, dtype, flags, alpha, epsilon)
    if backward:
      # the one difference: the backward kernels read beta element by element, so its alignment no longer matters
      want = _former_python_predicate(dtype, C, n_pix, alpha, epsilon, pow_alpha, pow_epsilon, x, ALIGNED, dy=dy)
    else:
      want = _former_python_predicate(dtype, C, n_pix, alpha, epsilon, pow_alpha, pow_epsilon, x, beta, boxes=C != 128)
    assert got == int(want), (backward, dtype, C, alpha, epsilon, pow_alpha, pow_epsilon, n_pix, x, beta, dy)
    checked += want
  assert (checked > 0) == (C != 64)
