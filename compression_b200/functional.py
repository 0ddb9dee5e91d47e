"""Functional CUDA entry points that have no op in the reference because the reference composes them from
TF primitives: GDN/IGDN forward + backward (``python/layers/gdn.py:371-421`` + TF autodiff) and the fused
quantise+encode / decode+dequantise paths of the entropy models."""
import ctypes as C

import torch

from compression_b200 import _lib
from compression_b200._lib import check

GDN_INVERSE = 1
GDN_RECTIFY = 2


def _stream() -> int:
  return torch.cuda.current_stream().cuda_stream


def _p(t):
  return None if t is None else C.c_void_p(t.data_ptr())


GDN_POW_ALPHA = 4      # trainable alpha: literal u ** alpha (no |u| / u^2 shortcut), gdn.py:380-388
GDN_POW_EPSILON = 8    # trainable epsilon: literal n ** epsilon, gdn.py:406-411


def _flags(inverse, rectify, pow_alpha=False, pow_epsilon=False):
  return ((GDN_INVERSE if inverse else 0) | (GDN_RECTIFY if rectify else 0) | (GDN_POW_ALPHA if pow_alpha else 0) |
          (GDN_POW_EPSILON if pow_epsilon else 0))


_IO16 = {torch.float16: 1, torch.bfloat16: 2}


def _gdn_args(x, gamma, beta):
  assert x.is_cuda and x.dtype in (torch.float32, torch.float16, torch.bfloat16)
  x = x.contiguous()
  C_ = x.shape[-1]
  gamma = gamma.to(device=x.device, dtype=torch.float32).contiguous()
  beta = beta.to(device=x.device, dtype=torch.float32).contiguous()
  assert gamma.shape == (C_, C_) and beta.shape == (C_,)
  return x, gamma, beta, C_, x.numel() // C_


def gdn_forward(x, gamma, beta, inverse=False, rectify=False, alpha=1.0, epsilon=1.0, pow_alpha=False,
                pow_epsilon=False):
  """x: float32 / float16 / bfloat16 CUDA [..., C] (channels-last, contiguous) -> y of the same shape and type."""
  x, gamma, beta, C_, n_pix = _gdn_args(x, gamma, beta)
  flags = _flags(inverse, rectify, pow_alpha, pow_epsilon)
  if x.dtype in _IO16:
    # 16-bit activations, float32 parameters and arithmetic (mixed precision, gdn_test.py:200-210): the kernel reads
    # and writes the 16-bit elements where the library has one for this call; otherwise convert
    if _lib.lib().tfcb_gdn_native_16bit(0, _p(x), _p(beta), None, n_pix, C_, _IO16[x.dtype], flags, float(alpha),
                                        float(epsilon)):
      y = torch.empty_like(x)
      check(_lib.lib().tfcb_gdn_forward_16bit(_p(x), _p(gamma), _p(beta), _p(y), n_pix, C_, _IO16[x.dtype], flags,
                                              float(alpha), float(epsilon), _stream()))
      return y
    return gdn_forward(x.float(), gamma, beta, inverse, rectify, alpha, epsilon, pow_alpha, pow_epsilon).to(x.dtype)
  y = torch.empty_like(x)
  check(_lib.lib().tfcb_gdn_forward(_p(x), _p(gamma), _p(beta), _p(y), n_pix, C_, flags, float(alpha), float(epsilon),
                                    _stream()))
  return y


def gdn_backward(x, gamma, beta, dy, inverse=False, rectify=False, alpha=1.0, epsilon=1.0, pow_alpha=False,
                 pow_epsilon=False):
  """Returns (dx, dgamma, dbeta) for upstream gradient dy; dx has x's type, dgamma / dbeta are float32."""
  x, gamma, beta, C_, n_pix = _gdn_args(x, gamma, beta)
  flags = _flags(inverse, rectify, pow_alpha, pow_epsilon)
  if x.dtype in _IO16:
    dy16 = dy.contiguous()
    if dy16.dtype == x.dtype and _lib.lib().tfcb_gdn_native_16bit(1, _p(x), _p(beta), _p(dy16), n_pix, C_, _IO16[x.dtype],
                                                                  flags, float(alpha), float(epsilon)):
      dx = torch.empty_like(x)
      dgamma = torch.empty_like(gamma)
      dbeta = torch.empty_like(beta)
      ws = torch.empty(int(_lib.lib().tfcb_gdn_backward_workspace_bytes(n_pix, C_)), dtype=torch.uint8, device=x.device)
      check(_lib.lib().tfcb_gdn_backward_16bit(_p(x), _p(gamma), _p(beta), _p(dy16), _p(dx), _p(dgamma), _p(dbeta),
                                               _p(ws), n_pix, C_, _IO16[x.dtype], flags, float(alpha), float(epsilon),
                                               _stream()))
      return dx, dgamma, dbeta
    # no native kernel (or a float32 dy, which keeps its precision): convert, run, hand dx back in x's type
    dx, dgamma, dbeta = gdn_backward(x.float(), gamma, beta, dy, inverse, rectify, alpha, epsilon, pow_alpha, pow_epsilon)
    return dx.to(x.dtype), dgamma, dbeta
  dy = dy.to(dtype=torch.float32).contiguous()
  dx = torch.empty_like(x)
  dgamma = torch.empty_like(gamma)
  dbeta = torch.empty_like(beta)
  ws_bytes = int(_lib.lib().tfcb_gdn_backward_workspace_bytes(n_pix, C_))
  ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
  check(_lib.lib().tfcb_gdn_backward(_p(x), _p(gamma), _p(beta), _p(dy), _p(dx), _p(dgamma), _p(dbeta), _p(ws),
                                     n_pix, C_, flags, float(alpha), float(epsilon), _stream()))
  return dx, dgamma, dbeta


def gdn_exponent_grads(x, gamma, beta, dy, inverse=False, rectify=False, alpha=1.0, epsilon=1.0, pow_alpha=True,
                       pow_epsilon=True):
  """(dL/dalpha, dL/depsilon) as a float32 [2] tensor: the gradients TF autodiff produces through `inputs ** alpha`
  and `norm_pool ** epsilon` when the exponents are trainable GDNParameters (gdn.py:345-367,388,411)."""
  x, gamma, beta, C_, n_pix = _gdn_args(x.float(), gamma, beta)
  dy = dy.to(dtype=torch.float32).contiguous()
  out = torch.empty(2, dtype=torch.float32, device=x.device)
  ws = torch.empty(int(_lib.lib().tfcb_gdn_exponent_grads_workspace_bytes()), dtype=torch.uint8, device=x.device)
  check(_lib.lib().tfcb_gdn_exponent_grads(_p(x), _p(gamma), _p(beta), _p(dy), _p(out), _p(ws), n_pix, C_,
                                           _flags(inverse, rectify, pow_alpha, pow_epsilon), float(alpha),
                                           float(epsilon), _stream()))
  return out


class _GDNFunction(torch.autograd.Function):
  """alpha_t / epsilon_t: 0-d tensors when the exponent is trainable (their value is read on the host: the kernels
  take the exponents as scalars), else None and the fixed value travels in `alpha` / `epsilon`."""

  @staticmethod
  def forward(ctx, x, gamma, beta, alpha_t, epsilon_t, inverse, rectify, alpha, epsilon):
    pa, pe = alpha_t is not None, epsilon_t is not None
    if pa:
      alpha = float(alpha_t)
    if pe:
      epsilon = float(epsilon_t)
    ctx.save_for_backward(x, gamma, beta)
    ctx.cfg = (inverse, rectify, alpha, epsilon, pa, pe)
    return gdn_forward(x, gamma, beta, inverse, rectify, alpha, epsilon, pa, pe)

  @staticmethod
  def backward(ctx, dy):
    x, gamma, beta = ctx.saved_tensors
    inverse, rectify, alpha, epsilon, pa, pe = ctx.cfg
    dx, dgamma, dbeta = gdn_backward(x, gamma, beta, dy, inverse, rectify, alpha, epsilon, pa, pe)
    dalpha = depsilon = None
    if (pa and ctx.needs_input_grad[3]) or (pe and ctx.needs_input_grad[4]):
      g2 = gdn_exponent_grads(x, gamma, beta, dy, inverse, rectify, alpha, epsilon, pa, pe)
      dalpha = g2[0] if pa else None
      depsilon = g2[1] if pe else None
    return dx, dgamma, dbeta, dalpha, depsilon, None, None, None, None


def gdn(x, gamma, beta, inverse=False, rectify=False, alpha=1.0, epsilon=1.0):
  """Differentiable GDN/IGDN on channels-last float32 / float16 / bfloat16 CUDA tensors (float32 parameters).  `alpha` / `epsilon`: Python numbers (fixed
  exponents: |u|, u^2, sqrt shortcuts and the tensor-core kernels apply) or 0-d tensors (trainable: literal pow, with
  gradients)."""
  at = alpha if isinstance(alpha, torch.Tensor) else None
  et = epsilon if isinstance(epsilon, torch.Tensor) else None
  return _GDNFunction.apply(x, gamma, beta, at, et, bool(inverse), bool(rectify),
                            1.0 if at is not None else float(alpha), 1.0 if et is not None else float(epsilon))


# ------------------------------------------------------------------------------------------------
# Fused quantise + encode / decode + dequantise (K3 fused into K4/K5 and K6)
# ------------------------------------------------------------------------------------------------
def _f32(t, device):
  return None if t is None else t.to(device=device, dtype=torch.float32).contiguous()


def _i32(t, device):
  return None if t is None else t.to(device=device, dtype=torch.int32).contiguous()


def encode_channel_f32(handle, y, quant_offset, cdf_offset):
  """symbols = int32(rint(y - quant_offset[c])) - cdf_offset[c] range-coded in channel mode, without
  materialising the int32 tensor (continuous_batched.py:375-382)."""
  handle._require()
  y = _f32(y, y.device)
  n = y.numel() // handle.n_streams
  check(_lib.lib().tfcb_encode_channel_f32(handle._h, _p(y), _p(_f32(quant_offset, y.device)),
                                           _p(_i32(cdf_offset, y.device)), n, _stream()))
  return handle


def encode_index_f32(handle, index, y, loc, cdf_offset):
  """symbols = int32(rint(y - loc)) - cdf_offset[index], index mode (continuous_indexed.py:378-385)."""
  handle._require()
  y = _f32(y, y.device)
  n = y.numel() // handle.n_streams
  check(_lib.lib().tfcb_encode_index_f32(handle._h, _p(_i32(index, y.device)), _p(y), _p(_f32(loc, y.device)),
                                         _p(_i32(cdf_offset, y.device)), n, _stream()))
  return handle


def decode_channel_f32(handle, out_shape, quant_offset, cdf_offset):
  """Decodes and dequantises: float(sym + cdf_offset[c]) + quant_offset[c] (continuous_batched.py:416-421)."""
  dev = handle._encoded.bytes_dev.device
  out = torch.empty(tuple(out_shape), dtype=torch.float32, device=dev)
  n = out.numel() // handle.n_streams
  check(_lib.lib().tfcb_decode_channel_f32(handle._h, _p(out), _p(_f32(quant_offset, dev)),
                                           _p(_i32(cdf_offset, dev)), n, _stream()))
  return out


def decode_index_f32(handle, index, loc, cdf_offset):
  """Decodes and dequantises in index mode (continuous_indexed.py:409-416)."""
  dev = handle._encoded.bytes_dev.device
  index = _i32(index, dev)
  out = torch.empty(tuple(index.shape), dtype=torch.float32, device=dev)
  n = out.numel() // handle.n_streams
  check(_lib.lib().tfcb_decode_index_f32(handle._h, _p(index), _p(out), _p(_f32(loc, dev)),
                                         _p(_i32(cdf_offset, dev)), n, _stream()))
  return out


def build_lookup(pmf, pmf_length, precision):
  """The per-row PMF -> CDF loop of _build_tables in one launch (continuous_base.py:282-294):
  pmf float32 [rows, max_len] (CUDA), pmf_length int [rows] -> 1-D int32 lookup [-p, cdf...]*rows."""
  import numpy as np
  pmf = pmf.to(dtype=torch.float32).contiguous()
  assert pmf.is_cuda and pmf.dim() == 2
  lens = np.ascontiguousarray(np.asarray(pmf_length.cpu() if isinstance(pmf_length, torch.Tensor) else pmf_length,
                                         dtype=np.int32).reshape(-1))
  assert lens.shape[0] == pmf.shape[0]
  total = int(lens.astype(np.int64).sum() + 3 * lens.shape[0])
  lookup = torch.empty(total, dtype=torch.int32, device=pmf.device)
  check(_lib.lib().tfcb_build_lookup(_p(pmf), pmf.shape[0], pmf.shape[1], lens.ctypes.data_as(C.c_void_p),
                                     int(precision), _p(lookup), _stream()))
  return lookup
