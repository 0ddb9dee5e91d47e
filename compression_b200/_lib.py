"""ctypes binding of libtfcb200.so (the C ABI declared in include/tfcb200.h).

The library is built in-tree (``make -C compression_b200/csrc`` or ``__graft_entry__.build()``).  There
is no CPU fallback: if the shared object is missing, loading fails loudly.
"""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TFCB_LIB_PATH") or os.path.join(_HERE, "libtfcb200.so")  # (override: kernel experiments)
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "tfcb200.h")

OK, INVALID_ARGUMENT, CUDA_ERROR, OUT_OF_MEMORY = 0, 1, 2, 3


class InvalidArgumentError(ValueError):
  """Analogue of tf.errors.InvalidArgumentError raised by the reference ops."""


class CudaError(RuntimeError):
  pass


def build(verbose: bool = False) -> str:
  """Compiles libtfcb200.so for sm_100a with nvcc (cross-compiles without a GPU)."""
  cmd = ["make", "-C", os.path.join(_HERE, "csrc"), "-j8"]
  if not verbose:
    cmd.insert(1, "-s")
  subprocess.run(cmd, check=True)
  return LIB_PATH


_p = C.POINTER
_vp, _i64, _i32, _int, _f32 = C.c_void_p, C.c_int64, C.c_int32, C.c_int, C.c_float

# name -> (restype, argtypes).  Mirrors include/tfcb200.h one to one; tests/test_abi.py checks that
# every prototype in the header is listed here and exported by the shared object.
SIGNATURES = {
    "tfcb_abi_version": (_int, []),
    "tfcb_last_error": (C.c_char_p, []),
    "tfcb_launch_count": (_i64, []),
    "tfcb_encoder_create": (_int, [_vp, _i64, _i64, _i64, _vp, _p(_vp)]),
    "tfcb_encode_channel": (_int, [_vp, _vp, _i64, _vp]),
    "tfcb_encode_index": (_int, [_vp, _vp, _vp, _i64, _vp]),
    "tfcb_encode_channel_f32": (_int, [_vp, _vp, _vp, _vp, _i64, _vp]),
    "tfcb_encode_index_f32": (_int, [_vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "tfcb_encoder_check": (_int, [_vp, _vp]),
    "tfcb_encode_finalize": (_int, [_vp, _vp, _p(_i64)]),
    "tfcb_encoder_output": (_int, [_vp, _p(_vp), _p(_vp)]),
    "tfcb_encoder_copy_output": (_int, [_vp, _vp, _vp, _vp]),
    "tfcb_encoder_destroy": (None, [_vp]),
    "tfcb_decoder_create": (_int, [_vp, _vp, _i64, _vp, _i64, _i64, _vp, _p(_vp)]),
    "tfcb_decode_channel": (_int, [_vp, _vp, _i64, _vp]),
    "tfcb_decode_index": (_int, [_vp, _vp, _vp, _i64, _vp]),
    "tfcb_decode_channel_f32": (_int, [_vp, _vp, _vp, _vp, _i64, _vp]),
    "tfcb_decode_index_f32": (_int, [_vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "tfcb_decode_finalize": (_int, [_vp, _vp, _vp]),
    "tfcb_decoder_destroy": (None, [_vp]),
    "tfcb_range_encode": (_int, [_vp, _vp, _int, _vp, _vp, _int, _int, _int, _vp, _i64, _p(_i64), _vp]),
    "tfcb_range_decode": (_int, [_vp, _i64, _vp, _int, _vp, _vp, _int, _int, _int, _vp, _vp]),
    "tfcb_pmf_to_quantized_cdf": (_int, [_vp, _i64, _i64, _int, _vp, _vp]),
    "tfcb_build_lookup": (_int, [_vp, _i64, _i64, _vp, _int, _vp, _vp]),
    "tfcb_run_length_encode": (_int, [_vp, _i64, _int, _int, _int, _vp, _i64, _p(_i64), _vp]),
    "tfcb_run_length_decode": (_int, [_vp, _i64, _int, _int, _int, _vp, _i64, _vp]),
    "tfcb_stochastic_round": (_int, [_vp, _int, _i64, _f32, _vp, _i64, _vp, _vp]),
    "tfcb_gdn_forward": (_int, [_vp, _vp, _vp, _vp, _i64, _int, _int, _f32, _f32, _vp]),
    "tfcb_gdn_forward_16bit": (_int, [_vp, _vp, _vp, _vp, _i64, _int, _int, _int, _f32, _f32, _vp]),
    "tfcb_gdn_backward_workspace_bytes": (_i64, [_i64, _int]),
    "tfcb_gdn_exponent_grads_workspace_bytes": (_i64, []),
    "tfcb_gdn_exponent_grads": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _f32, _f32, _vp]),
    "tfcb_gdn_backward": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _f32, _f32, _vp]),
    "tfcb_gdn_backward_16bit": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _int, _f32, _f32, _vp]),
    "tfcb_gdn_native_16bit": (_int, [_int, _vp, _vp, _vp, _i64, _int, _int, _int, _f32, _f32]),
}

_lib = None


def lib():
  """Returns the loaded CDLL; raises if the CUDA extension has not been built."""
  global _lib
  if _lib is None:
    if not os.path.exists(LIB_PATH):
      raise ImportError(
          f"{LIB_PATH} is missing. compression_b200 has no CPU fallback: build the CUDA library with "
          "`python -c 'import __graft_entry__ as g; g.build()'` or `make -C compression_b200/csrc`.")
    handle = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
      fn = getattr(handle, name)
      fn.restype = res
      fn.argtypes = args
    if handle.tfcb_abi_version() != 1:
      raise ImportError("libtfcb200.so ABI version mismatch")
    _lib = handle
  return _lib


def last_error() -> str:
  return (lib().tfcb_last_error() or b"").decode()


def check(rc: int) -> None:
  if rc == OK:
    return
  msg = last_error()
  if rc == INVALID_ARGUMENT:
    raise InvalidArgumentError(msg)
  if rc == OUT_OF_MEMORY:
    raise MemoryError(msg)
  raise CudaError(msg)


def launch_count() -> int:
  return int(lib().tfcb_launch_count())
