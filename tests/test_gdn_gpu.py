"""GPU parity for GDN/IGDN: closed forms of the reference's tests (layers/gdn_test.py:42-88, atol 1e-6) and
random-parameter parity against the fp64 oracle (north-star tolerance: 1e-5 relative)."""
import numpy as np
import pytest
import torch

from oracle import gdn_oracle

pytestmark = pytest.mark.gpu

RTOL = 1e-5  # BASELINE.json north_star: "GDN within 1e-5 relative of the reference fp32 path"


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
  return torch.randn(n_pix, C, generator=g) * scale


def _relerr(got, want):
  want = want.double()
  return ((got.double().cpu() - want).abs() / (want.abs() + 1e-30)).max().item()


@pytest.mark.parametrize("C", [3, 5, 32, 128, 192])
def test_closed_forms(F, C):
  x = torch.rand(77, C).cuda() - 0.5
  eye = (0.1 * torch.eye(C)).cuda()
  ones = torch.ones(C).cuda()
  xc = x.cpu()
  y = F.gdn_forward(x, eye, ones).cpu()
  assert torch.allclose(y, xc / (1 + 0.1 * xc.abs()), rtol=0, atol=1e-6)
  y = F.gdn_forward(x, eye, ones, inverse=True).cpu()
  assert torch.allclose(y, xc * (1 + 0.1 * xc.abs()), rtol=0, atol=1e-6)
  y = F.gdn_forward(x, eye, ones, rectify=True).cpu()
  xr = torch.relu(xc)
  assert torch.allclose(y, xr / (1 + 0.1 * xr), rtol=0, atol=1e-6)
  y = F.gdn_forward(x, eye, ones, alpha=2, epsilon=0.5).cpu()
  assert torch.allclose(y, xc / torch.sqrt(1 + 0.1 * xc**2), rtol=0, atol=1e-6)
  # fixed gamma = all ones, beta = 0 (gdn_test.py:80-88)
  y = F.gdn_forward(x.abs() + 0.1, torch.ones(C, C).cuda(), torch.zeros(C).cuda()).cpu()
  xa = xc.abs() + 0.1
  assert torch.allclose(y, xa / xa.sum(-1, keepdim=True), rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("C,n_pix", [(128, 4099), (128, 1), (128, 129), (128, 128 * 148 * 3 + 5), (192, 2500),
                                     (192, 128 * 148 * 2 + 9), (64, 333), (7, 129)])
@pytest.mark.parametrize("inverse", [False, True])
def test_forward_vs_fp64_oracle(F, C, n_pix, inverse):
  gamma, beta = _params(C, 4)
  x = _x(n_pix, C, 6)
  want = gdn_oracle.gdn_reference(x, gamma, beta, inverse=inverse)
  got = F.gdn_forward(x.cuda(), gamma.cuda(), beta.cuda(), inverse=inverse)
  assert _relerr(got, want) < RTOL


@pytest.mark.parametrize("alpha,epsilon,rectify", [(1, 1, True), (2, 0.5, False), (1.5, 0.7, True), (2, 1, False),
                                                   (1, 0.5, False)])
@pytest.mark.parametrize("C", [64, 128])  # 64: fp32 kernels, 128: tensor-core kernel's general (non-FAST) variant
def test_forward_variants(F, C, alpha, epsilon, rectify):
  gamma, beta = _params(C, 5)
  x = _x(1000, C, 8)
  for inverse in (False, True):
    want = gdn_oracle.gdn_reference(x, gamma, beta, inverse, rectify, alpha, epsilon)
    got = F.gdn_forward(x.cuda(), gamma.cuda(), beta.cuda(), inverse, rectify, alpha, epsilon)
    mask = torch.isfinite(want)
    err = ((got.double().cpu() - want)[mask].abs() / (want[mask].abs() + 1e-6)).max().item()
    assert err < 2e-5


@pytest.mark.parametrize("C,n_pix", [(128, 3000), (128, 1), (128, 129), (128, 128 * 148 * 2 + 77), (192, 1111), (192, 1),
                                     (192, 128 * 148 * 2 + 300), (5, 257)])
@pytest.mark.parametrize("inverse", [False, True])
def test_backward_vs_fp64_oracle(F, C, n_pix, inverse):
  gamma, beta = _params(C, 14)
  x = _x(n_pix, C, 16)
  dy = torch.randn(n_pix, C, generator=torch.Generator().manual_seed(1))
  wx, wg, wb = gdn_oracle.gdn_reference_grads(x, gamma, beta, dy, inverse=inverse)
  dx, dg, db = F.gdn_backward(x.cuda(), gamma.cuda(), beta.cuda(), dy.cuda(), inverse=inverse)

  def close(got, want, tol):
    scale = want.abs().max().item()
    return ((got.double().cpu() - want).abs().max().item() / scale) < tol

  assert close(dx, wx, 2e-5)
  assert close(dg, wg, 2e-5)
  assert close(db, wb, 2e-5)


@pytest.mark.parametrize("C", [64, 128, 192])
@pytest.mark.parametrize("alpha,epsilon,rectify", [(1, 1, True), (2, 0.5, False), (2, 1, False), (1, 0.5, False),
                                                   (1.5, 0.7, True)])
# 700 pixels are 6 tiles, one per CTA; 297 tiles give every CTA of a 148-SM grid a second tile (dgamma flushes)
@pytest.mark.parametrize("n_pix", [700, 128 * 148 * 2 + 77])
def test_backward_variants(F, C, alpha, epsilon, rectify, n_pix):
  gamma, beta = _params(C, 21)
  x = _x(n_pix, C, 22)
  dy = torch.randn(n_pix, C, generator=torch.Generator().manual_seed(23))
  for inverse in (False, True):
    wx, wg, wb = gdn_oracle.gdn_reference_grads(x, gamma, beta, dy, inverse, rectify, alpha, epsilon)
    dx, dg, db = F.gdn_backward(x.cuda(), gamma.cuda(), beta.cuda(), dy.cuda(), inverse, rectify, alpha, epsilon)
    for got, want in ((dx, wx), (dg, wg), (db, wb)):
      want = torch.nan_to_num(want, nan=0.0, posinf=0.0, neginf=0.0)
      scale = want.abs().max().item()
      assert ((got.double().cpu() - want).abs().max().item() / scale) < 3e-5


def test_autograd_wrapper(F):
  C = 32
  gamma, beta = _params(C, 2)
  x = _x(100, C, 3).cuda().requires_grad_(True)
  g = gamma.cuda().requires_grad_(True)
  b = beta.cuda().requires_grad_(True)
  y = F.gdn(x, g, b)
  y.square().sum().backward()
  assert x.grad is not None and g.grad.shape == (C, C) and b.grad.shape == (C,)


def _err_report(got, want):
  """(max |err| / max |want|,  max elementwise relative error over entries with |want| >= 1e-2 max |want|)."""
  got, want = got.double().cpu(), want.double()
  scale = want.abs().max().item()
  err = (got - want).abs()
  big = want.abs() >= 1e-2 * scale
  return err.max().item() / scale, (err[big] / want.abs()[big]).max().item()


@pytest.mark.parametrize("C,n_pix", [(128, 2 * 1024 * 1024 + 77), (192, 2 * 1024 * 1024 + 300)])
def test_backward_at_two_million_pixels_vs_fp64_oracle(F, C, n_pix):
  """dgamma / dbeta reduce over every pixel (148 per-CTA partials x thousands of tiles): the accumulation error
  must not grow past the contract at training-sized inputs.  Bounds asserted: every gradient within 1e-5 of its
  largest entry (the contract's 1e-5, on the scale that does not blow up where a gradient cancels to ~0; measured
  2.6e-6 / 5.3e-6 / 1.9e-6 for dx / dgamma / dbeta at C = 128, 2.5e-6 / 4.3e-6 / 1.5e-6 at C = 192), and elementwise
  within 5e-4 relative on entries >= 1 % of the largest (measured: dx 9.4e-5, dgamma 2.9e-4 -- every gradient is a
  signed sum, so an entry at 1 % of the maximum carries the absolute error of the large ones; the fp32 reference
  path itself, the same graph in torch fp32 on the CPU, is printed beside it: 5e-7 of max, 2e-5 elementwise).
  Before the periodic flush of the TMEM accumulator (kDgFlush, gdn_tc.cu) dgamma drifted to 6e-5 of max here."""
  gamma, beta = _params(C, 31)
  x = _x(n_pix, C, 32)
  dy = torch.randn(n_pix, C, generator=torch.Generator().manual_seed(33))
  wx, wg, wb = gdn_oracle.gdn_reference_grads(x, gamma, beta, dy)
  dx, dg, db = F.gdn_backward(x.cuda(), gamma.cuda(), beta.cuda(), dy.cuda())
  rep = {name: _err_report(g, w) for name, g, w in (("dx", dx, wx), ("dgamma", dg, wg), ("dbeta", db, wb))}
  fx, fg, fb = gdn_oracle.gdn_reference_grads(x, gamma, beta, dy, dtype=torch.float32)
  ref32 = {name: _err_report(g, w) for name, g, w in (("dx", fx, wx), ("dgamma", fg, wg), ("dbeta", fb, wb))}
  print(f"GDN backward C={C} n_pix={n_pix}: (max err / max |want|, max elementwise rel. err where |want| >= 1% of max)"
        f" CUDA = {rep}; torch-CPU fp32 reference path = {ref32}")
  for name, (of_max, rel) in rep.items():
    assert of_max < 1e-5, (name, of_max)
    assert rel < 5e-4, (name, rel)
  # forward at the same size, elementwise
  want = gdn_oracle.gdn_reference(x, gamma, beta)
  got = F.gdn_forward(x.cuda(), gamma.cuda(), beta.cuda())
  assert _relerr(got, want) < RTOL


def _graph64(x, gamma, beta, alpha, epsilon, inverse, rectify, pow_alpha, pow_epsilon):
  """gdn.py:377-415 in float64; alpha / epsilon None-able shortcuts as in the reference."""
  u = torch.relu(x) if rectify else x
  if not pow_alpha and float(alpha) == 1:
    pool = u if rectify else u.abs()
  elif not pow_alpha and float(alpha) == 2:
    pool = u.square()
  else:
    pool = u**alpha
  n = pool @ gamma + beta
  if not pow_epsilon and float(epsilon) == 1:
    pass
  elif not pow_epsilon and float(epsilon) == .5:
    n = n.sqrt()
  else:
    n = n**epsilon
  return u * n if inverse else u / n


@pytest.mark.parametrize("C,n_pix", [(5, 300), (32, 1000), (128, 3000)])
@pytest.mark.parametrize("alpha,epsilon,train_a,train_e,rectify,inverse", [
    (1.3, 1.0, True, False, True, False), (1.0, 0.8, False, True, False, False), (1.3, 0.8, True, True, True, False),
    (2.0, 0.6, False, True, False, True), (1.0, 1.0, True, True, True, True)])
def test_trainable_exponents_vs_fp64_graph(F, C, n_pix, alpha, epsilon, train_a, train_e, rectify, inverse):
  """gdn.py:345-367: alpha / epsilon as trainable parameters.  Forward and all five gradients (x, gamma, beta, alpha,
  epsilon) come from the CUDA kernels (literal pow + the exponent-gradient kernel) and agree with the reference's
  graph differentiated by autograd in float64; a FIXED exponent of a mixed configuration keeps its |u| / u^2 / sqrt
  shortcut (gdn.py:380-388), a trainable one sitting at 1.0 does not."""
  gamma, beta = _params(C, 31)
  x = (_x(n_pix, C, 32) * 1.5).cuda().requires_grad_(True)
  g = gamma.cuda().requires_grad_(True)
  b = beta.cuda().requires_grad_(True)
  a_t = torch.tensor(alpha, device="cuda", requires_grad=True) if train_a else alpha
  e_t = torch.tensor(epsilon, device="cuda", requires_grad=True) if train_e else epsilon
  y = F.gdn(x, g, b, inverse, rectify, a_t, e_t)
  dy = torch.randn(n_pix, C, generator=torch.Generator().manual_seed(33)).cuda()
  leaves = [x, g, b] + ([a_t] if train_a else []) + ([e_t] if train_e else [])
  got = torch.autograd.grad(y, leaves, dy)
  x64, g64, b64 = (t.detach().double().requires_grad_(True) for t in (x, g, b))
  a64 = torch.tensor(alpha, dtype=torch.float64, device="cuda", requires_grad=True) if train_a else alpha
  e64 = torch.tensor(epsilon, dtype=torch.float64, device="cuda", requires_grad=True) if train_e else epsilon
  y64 = _graph64(x64, g64, b64, a64, e64, inverse, rectify, train_a, train_e)
  want = torch.autograd.grad(y64, [x64, g64, b64] + ([a64] if train_a else []) + ([e64] if train_e else []), dy.double())
  assert float(((y.double() - y64).abs() / (y64.abs() + 1e-6)).max()) < 2e-5
  for gt, w in zip(got, want):
    w = torch.nan_to_num(w, nan=0.0, posinf=0.0, neginf=0.0)
    scale = float(w.abs().max()) + 1e-12
    assert float((gt.double() - w).abs().max()) / scale < 1e-4, (tuple(gt.shape), float((gt.double() - w).abs().max()), scale)


def test_layer_with_trainable_exponents_uses_the_kernels(tfc_mod=None):
  import compression_b200 as tfc
  from compression_b200 import _lib
  layer = tfc.GDN(alpha_parameter=None, epsilon_parameter=None, rectify=True)
  x = torch.rand(200, 16).cuda() + 0.1
  n0 = _lib.launch_count()
  y = layer(x)
  y.square().sum().backward()
  assert _lib.launch_count() >= n0 + 3
  grads = {n: p.grad for n, p in layer.named_parameters()}
  assert len(grads) == 4 and all(v is not None and torch.isfinite(v).all() for v in grads.values())


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("n_pix", [1, 129, 128 * 148 * 2 + 5])
@pytest.mark.parametrize("inverse,alpha,epsilon,rectify", [(False, 1, 1, False), (True, 1, 1, False), (False, 2, 0.5, False),
                                                           (False, 1, 1, True)])
def test_sixteen_bit_activations_native_kernel(F, dtype, n_pix, inverse, alpha, epsilon, rectify):
  """Mixed precision (gdn_test.py:200-210): x, y in 16 bits, float32 parameters.  The C = 128 kernel reads and writes the
  16-bit elements itself; its result is the float32 result of the same (already rounded) inputs, rounded once."""
  from compression_b200 import _lib
  C = 128
  gamma, beta = _params(C, 41)
  x = _x(n_pix, C, 42).to(dtype).cuda()
  n0 = _lib.launch_count()
  y = F.gdn_forward(x, gamma.cuda(), beta.cuda(), inverse, rectify, alpha, epsilon)
  assert _lib.launch_count() == n0 + 1 and y.dtype == dtype  # one kernel, no conversion passes
  # it is exactly the float32 kernel's output (same inputs) rounded to the activation type ...
  y32 = F.gdn_forward(x.float(), gamma.cuda(), beta.cuda(), inverse, rectify, alpha, epsilon)
  assert torch.equal(y, y32.to(dtype))
  # ... i.e. within half an ulp of the activation type of the float64 oracle (normal range of float16)
  want = gdn_oracle.gdn_reference(x.float().cpu(), gamma, beta, inverse, rectify, alpha, epsilon)
  eps_io = 2.0**-11 if dtype == torch.float16 else 2.0**-8
  big = want.abs() >= 1e-3
  err = ((y.double().cpu() - want).abs() / (want.abs() + 1e-30))[big].max().item() if bool(big.any()) else 0.0
  assert err <= eps_io * 1.01 + 2e-5


def test_sixteen_bit_module_and_gradients(F):
  import compression_b200 as tfc
  layer = tfc.GDN()
  x = (torch.randn(500, 128) * 2).to(torch.bfloat16).cuda().requires_grad_(True)
  y = layer(x)
  assert y.dtype == torch.bfloat16
  for p in layer.parameters():
    assert p.dtype == torch.float32  # gdn_test.py:205-206
  y.float().square().sum().backward()
  assert x.grad is not None and x.grad.dtype == torch.bfloat16
  # other widths convert and still return the activation type
  y2 = tfc.GDN()(torch.randn(70, 192).half().cuda())
  assert y2.dtype == torch.float16
