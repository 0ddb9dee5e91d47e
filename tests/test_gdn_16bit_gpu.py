"""16-bit GDN activations (mixed precision, gdn_test.py:200-210: float32 variables, float16 / bfloat16 activations).

The kernels that read and write 16-bit x, dy, y and dx themselves (C = 192 forward, C = 128 and C = 192 backward) must
give exactly what the float32 kernels give on the widened inputs, rounded once to the activation type; dgamma / dbeta
(float32 outputs, summed with shared-memory and global atomics) agree to the last bits.  Calls without a native kernel
keep converting to float32."""
import copy

import pytest
import torch

from oracle import gdn_oracle

DTYPES = [torch.float16, torch.bfloat16]
HALF_ULP = {torch.float16: 2.0**-11, torch.bfloat16: 2.0**-8}  # relative, normal range


@pytest.fixture(scope="module")
def F():
  from compression_b200 import functional
  return functional


def _params(C, seed):
  g = torch.Generator().manual_seed(seed)
  gamma = 0.1 * torch.eye(C) + (0.02 * torch.randn(C, C, generator=g)).abs()
  beta = 1.0 + 0.5 * torch.rand(C, generator=g)
  return gamma, beta


def _x(n_pix, C, seed):
  g = torch.Generator().manual_seed(seed)
  scale = 0.05 + 3.95 * torch.rand(C, generator=g)
  x = torch.randn(n_pix, C, generator=g) * scale
  x[::7, ::5] = 0.0  # exact zeros: sign(0) = 0 and the rectifier's edge
  return x


def _dy(n_pix, C, seed):
  return torch.randn(n_pix, C, generator=torch.Generator().manual_seed(seed))


def _of_max(got, want):
  want = torch.nan_to_num(want.double().cpu(), nan=0.0, posinf=0.0, neginf=0.0)
  return (got.double().cpu() - want).abs().max().item() / want.abs().max().item()


# ------------------------------------------------------------------------------------------------
# Forward, C = 192
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n_pix", [1, 129, 2500, 128 * 148 * 2 + 9])
@pytest.mark.parametrize("inverse", [False, True])
@pytest.mark.parametrize("alpha,epsilon,rectify", [(1, 1, False), (2, 0.5, False), (1, 1, True)])
def test_forward_c192(F, dtype, n_pix, inverse, alpha, epsilon, rectify):
  C = 192
  gamma, beta = _params(C, 51)
  x = _x(n_pix, C, 52).to(dtype).cuda()
  g, b = gamma.cuda(), beta.cuda()
  y = F.gdn_forward(x, g, b, inverse, rectify, alpha, epsilon)
  assert y.dtype == dtype and y.shape == x.shape
  # exactly the float32 kernel's output on the widened input, rounded once ...
  y32 = F.gdn_forward(x.float(), g, b, inverse, rectify, alpha, epsilon)
  assert torch.equal(y, y32.to(dtype))
  # ... i.e. within half an ulp of the activation type of the float64 oracle (normal range of float16)
  want = gdn_oracle.gdn_reference(x.float().cpu(), gamma, beta, inverse, rectify, alpha, epsilon)
  big = want.abs() >= 1e-3
  err = ((y.double().cpu() - want).abs() / (want.abs() + 1e-30))[big].max().item() if bool(big.any()) else 0.0
  assert err <= HALF_ULP[dtype] * 1.01 + 2e-5


# ------------------------------------------------------------------------------------------------
# Backward, C = 128 and C = 192
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("C", [128, 192])
# 700 pixels are 6 tiles, one per CTA; 297 tiles give every CTA of a 148-SM grid a second tile (dgamma flushes)
@pytest.mark.parametrize("n_pix", [1, 700, 128 * 148 * 2 + 77])
@pytest.mark.parametrize("inverse", [False, True])
@pytest.mark.parametrize("alpha,epsilon,rectify", [(1, 1, False), (1, 1, True), (2, 0.5, False), (2, 1, False)])
def test_backward(F, dtype, C, n_pix, inverse, alpha, epsilon, rectify):
  gamma, beta = _params(C, 61)
  x = _x(n_pix, C, 62).to(dtype)
  dy = _dy(n_pix, C, 63).to(dtype)
  g, b = gamma.cuda(), beta.cuda()
  dx, dg, db = F.gdn_backward(x.cuda(), g, b, dy.cuda(), inverse, rectify, alpha, epsilon)
  assert dx.dtype == dtype and dg.dtype == torch.float32 and db.dtype == torch.float32
  # the float32 kernels on the widened x and dy
  dx32, dg32, db32 = F.gdn_backward(x.float().cuda(), g, b, dy.float().cuda(), inverse, rectify, alpha, epsilon)
  assert torch.equal(dx, dx32.to(dtype))
  assert _of_max(dg, dg32) <= 1e-6
  assert _of_max(db, db32) <= 1e-6
  # the float64 oracle on the widened inputs: dgamma / dbeta as the float32 path is held to; dx additionally carries
  # the one rounding to the activation type (half an ulp of the entry)
  wx, wg, wb = gdn_oracle.gdn_reference_grads(x.float(), gamma, beta, dy.float(), inverse, rectify, alpha, epsilon)
  assert _of_max(dg, wg) < 3e-5
  assert _of_max(db, wb) < 3e-5
  wx = torch.nan_to_num(wx, nan=0.0, posinf=0.0, neginf=0.0)
  err = (dx.double().cpu() - wx).abs()
  assert bool((err <= HALF_ULP[dtype] * 1.01 * wx.abs() + 3e-5 * wx.abs().max()).all())


# ------------------------------------------------------------------------------------------------
# No conversion passes: launches and memory
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("C", [128, 192])
def test_no_conversion_passes(F, dtype, C):
  from compression_b200 import _lib
  n_pix = 65536 + 77
  gamma, beta = _params(C, 71)
  g, b = gamma.cuda(), beta.cuda()
  x = _x(n_pix, C, 72).to(dtype).cuda()
  dy = _dy(n_pix, C, 73).to(dtype).cuda()
  x32, dy32 = x.float(), dy.float()
  elem = n_pix * C

  def run(fn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    n0 = _lib.launch_count()
    out = fn()
    torch.cuda.synchronize()
    return _lib.launch_count() - n0, torch.cuda.max_memory_allocated() - base, out

  ws = int(_lib.lib().tfcb_gdn_backward_workspace_bytes(n_pix, C))
  slack = 1 << 20
  if C == 192:  # (the C = 128 forward already had a native kernel)
    launches, peak, _ = run(lambda: F.gdn_forward(x, g, b))
    launches32, _, _ = run(lambda: F.gdn_forward(x32, g, b))
    assert launches == launches32
    assert peak <= 2 * elem + slack  # y; the conversion path would add x and y in float32, 8 B/element
  launches, peak, _ = run(lambda: F.gdn_backward(x, g, b, dy))
  launches32, _, _ = run(lambda: F.gdn_backward(x32, g, b, dy32))
  assert launches == launches32
  # dx, dgamma, dbeta, the workspace; the conversion path would add x, dy and dx in float32, 12 B/element
  assert peak <= 2 * elem + 4 * (C * C + C) + ws + slack


# ------------------------------------------------------------------------------------------------
# The module: 16-bit activations in, 16-bit activations and float32 parameter gradients out
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("inverse", [False, True])
def test_module_bfloat16_c192(inverse):
  import compression_b200 as tfc
  torch.manual_seed(81)
  x32 = torch.randn(2, 33, 40, 192, device="cuda") * 2
  x = x32.to(torch.bfloat16).requires_grad_(True)
  layer = tfc.GDN(inverse=inverse)
  y = layer(x)
  layer32 = copy.deepcopy(layer)
  assert y.dtype == torch.bfloat16
  dy = torch.randn(y.shape, generator=torch.Generator().manual_seed(82)).to(torch.bfloat16).cuda()
  y.backward(dy)
  assert x.grad is not None and x.grad.dtype == torch.bfloat16
  xw = x.detach().float().requires_grad_(True)
  y32 = layer32(xw)
  assert torch.equal(y, y32.to(torch.bfloat16))
  y32.backward(dy.float())
  assert torch.equal(x.grad, xw.grad.to(torch.bfloat16))
  params = dict(layer.named_parameters())
  params32 = dict(layer32.named_parameters())
  assert params.keys() == params32.keys() and params
  for name, p in params.items():
    assert p.dtype == torch.float32 and p.grad.dtype == torch.float32
    assert _of_max(p.grad, params32[name].grad) <= 1e-6, name


# ------------------------------------------------------------------------------------------------
# Calls without a native kernel still convert, with unchanged results
# ------------------------------------------------------------------------------------------------
def _misaligned(n_pix, C, dtype, src):
  t = torch.empty(n_pix * C + 1, dtype=dtype, device="cuda")[1:].view(n_pix, C)
  t.copy_(src)
  assert t.data_ptr() % 16 != 0
  return t


@pytest.mark.gpu
@pytest.mark.parametrize("C", [128, 192])
def test_misaligned_view_takes_the_conversion_path(F, C):
  n_pix = 500
  gamma, beta = _params(C, 91)
  g, b = gamma.cuda(), beta.cuda()
  dtype = torch.bfloat16
  x = _misaligned(n_pix, C, dtype, _x(n_pix, C, 92).to(dtype))
  dy = _misaligned(n_pix, C, dtype, _dy(n_pix, C, 93).to(dtype))
  y = F.gdn_forward(x, g, b)
  assert torch.equal(y, F.gdn_forward(x.float(), g, b).to(dtype))
  dx, dg, db = F.gdn_backward(x, g, b, dy)
  dx32, dg32, db32 = F.gdn_backward(x.float(), g, b, dy.float())
  assert torch.equal(dx, dx32.to(dtype))
  assert _of_max(dg, dg32) <= 1e-6 and _of_max(db, db32) <= 1e-6  # (C = 128 sums dbeta with shared-memory atomics)


@pytest.mark.gpu
@pytest.mark.parametrize("C", [128, 192])
def test_misaligned_beta_keeps_the_native_backward(F, C):
  """The backward kernels read beta element by element, so a beta view off a 16-byte boundary does not send a 16-bit
  backward through the conversion path (the forward's C = 128 kernel reads beta with 16-byte loads and still does)."""
  from compression_b200 import _lib
  n_pix = 65536 + 77
  gamma, beta = _params(C, 121)
  g = gamma.cuda()
  b = torch.empty(C + 1, device="cuda")[1:]
  b.copy_(beta)
  assert b.data_ptr() % 16 != 0
  dtype = torch.bfloat16
  x = _x(n_pix, C, 122).to(dtype).cuda()
  dy = _dy(n_pix, C, 123).to(dtype).cuda()
  ws = int(_lib.lib().tfcb_gdn_backward_workspace_bytes(n_pix, C))
  torch.cuda.synchronize()
  torch.cuda.reset_peak_memory_stats()
  base = torch.cuda.memory_allocated()
  dx, dg, db = F.gdn_backward(x, g, b, dy)
  torch.cuda.synchronize()
  # dx, dgamma, dbeta, the workspace; the conversion path would add x, dy and dx in float32, 12 B/element
  assert torch.cuda.max_memory_allocated() - base <= 2 * n_pix * C + 4 * (C * C + C) + ws + (1 << 20)
  dx32, dg32, db32 = F.gdn_backward(x.float(), g, b, dy.float())
  assert torch.equal(dx, dx32.to(dtype))
  assert _of_max(dg, dg32) <= 1e-6 and _of_max(db, db32) <= 1e-6  # (C = 128 sums dbeta with shared-memory atomics)


@pytest.mark.gpu
def test_float32_dy_keeps_its_precision(F):
  C, n_pix = 192, 700
  gamma, beta = _params(C, 101)
  g, b = gamma.cuda(), beta.cuda()
  x = _x(n_pix, C, 102).to(torch.bfloat16).cuda()
  dy = _dy(n_pix, C, 103).cuda()  # float32: not rounded to bfloat16
  dx, dg, db = F.gdn_backward(x, g, b, dy)
  dx32, dg32, db32 = F.gdn_backward(x.float(), g, b, dy)
  assert dx.dtype == torch.bfloat16
  assert torch.equal(dx, dx32.to(torch.bfloat16))
  assert _of_max(dg, dg32) <= 1e-6 and _of_max(db, db32) <= 1e-6  # (C = 128 sums dbeta with shared-memory atomics)


@pytest.mark.gpu
@pytest.mark.parametrize("C,alpha", [(64, 1.0), (192, torch.tensor(1.0))])  # other C; trainable alpha
def test_configurations_without_a_native_kernel(F, C, alpha):
  n_pix = 300
  gamma, beta = _params(C, 111)
  g, b = gamma.cuda(), beta.cuda()
  x = _x(n_pix, C, 112).to(torch.float16).cuda()
  dy = _dy(n_pix, C, 113).to(torch.float16).cuda()
  pa = isinstance(alpha, torch.Tensor)
  a = float(alpha)
  y = F.gdn_forward(x, g, b, alpha=a, pow_alpha=pa)
  assert y.dtype == torch.float16
  assert torch.equal(y, F.gdn_forward(x.float(), g, b, alpha=a, pow_alpha=pa).to(torch.float16))
  dx, dg, db = F.gdn_backward(x, g, b, dy, alpha=a, pow_alpha=pa)
  dx32, dg32, db32 = F.gdn_backward(x.float(), g, b, dy.float(), alpha=a, pow_alpha=pa)
  assert torch.equal(dx, dx32.to(torch.float16))
  assert _of_max(dg, dg32) <= 1e-6 and _of_max(db, db32) <= 1e-6  # (C = 128 sums dbeta with shared-memory atomics)


# ------------------------------------------------------------------------------------------------
# Host-side argument checks (no device needed)
# ------------------------------------------------------------------------------------------------
def test_sixteen_bit_entries_reject_bad_arguments_without_a_device():
  from compression_b200 import _lib
  lib = _lib.lib()
  fake = 1 << 20  # never dereferenced: every call below fails before it touches the device
  ws = fake
  for dtype in (0, 3):
    with pytest.raises(_lib.InvalidArgumentError, match="dtype"):
      _lib.check(lib.tfcb_gdn_backward_16bit(fake, fake, fake, fake, fake, fake, fake, ws, 256, 128, dtype, 0, 1.0, 1.0,
                                             None))
    with pytest.raises(_lib.InvalidArgumentError, match="dtype"):
      _lib.check(lib.tfcb_gdn_forward_16bit(fake, fake, fake, fake, 256, 128, dtype, 0, 1.0, 1.0, None))
  with pytest.raises(_lib.InvalidArgumentError, match="native 16-bit"):
    _lib.check(lib.tfcb_gdn_backward_16bit(fake, fake, fake, fake, fake, fake, fake, ws, 256, 64, 2, 0, 1.0, 1.0, None))
  with pytest.raises(_lib.InvalidArgumentError, match="native 16-bit"):
    _lib.check(lib.tfcb_gdn_forward_16bit(fake, fake, fake, fake, 256, 64, 2, 0, 1.0, 1.0, None))
  with pytest.raises(_lib.InvalidArgumentError, match="null pointer"):
    _lib.check(lib.tfcb_gdn_backward_16bit(fake, fake, fake, None, fake, fake, fake, ws, 256, 128, 1, 0, 1.0, 1.0, None))
  with pytest.raises(_lib.InvalidArgumentError, match="null pointer"):
    _lib.check(lib.tfcb_gdn_forward_16bit(None, fake, fake, fake, 256, 192, 1, 0, 1.0, 1.0, None))
  with pytest.raises(_lib.InvalidArgumentError, match="bad GDN shape"):
    _lib.check(lib.tfcb_gdn_backward_16bit(fake, fake, fake, fake, fake, fake, fake, ws, -1, 128, 1, 0, 1.0, 1.0, None))
