"""GPU parity for the legacy ops, PmfToQuantizedCdf and GDN (first slice; widened in later files)."""
import numpy as np
import pytest
import torch

import golden_util
import oracle
import util

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
  from compression_b200 import gen_ops
  return gen_ops


# ---- legacy RangeEncode / RangeDecode: range_coding_kernels_test.cc:246-322 shapes ----
@pytest.mark.parametrize("dshape,cshape,precision", [
    ((1, 32, 32, 16), (1, 32, 32, 16, 33), 14),   # NoBroadcast
    ((1, 64, 64), (1, 1, 1, 30), 9),              # Broadcast over all axes
    ((2, 16, 32, 7), (1, 1, 1, 7, 21), 13),       # per-channel
    ((2, 8, 16, 7), (2, 1, 16, 1, 12), 10),       # alternating pattern
    ((37,), (1, 5), 6),
])
def test_legacy_roundtrip_matches_oracle(ops, dshape, cshape, precision):
  rng = np.random.default_rng(sum(dshape))
  O = oracle.best()
  nb = cshape[-1] - 1
  rows = int(np.prod(cshape[:-1]))
  cdf = np.stack([util.random_cdf(rng, nb, precision, peaky=3) for _ in range(rows)]).reshape(cshape)
  data = rng.integers(0, nb, size=dshape).astype(np.int16)
  want = O.range_encode(data, cdf, precision)
  got = ops.range_encode(torch.from_numpy(data).cuda(), torch.from_numpy(cdf).cuda(), precision)
  assert got == want
  dec = ops.range_decode(want, list(dshape), torch.from_numpy(cdf).cuda(), precision)
  assert dec.dtype == torch.int16
  assert np.array_equal(dec.cpu().numpy(), data)
  assert np.array_equal(O.range_decode(got, dshape, cdf, precision), data)


def test_legacy_errors(ops):
  cdf = torch.tensor([[0, 16, 18, 32]], dtype=torch.int32).cuda()  # range_coding_kernels_test.cc:454
  data = torch.tensor([0, 1, 2], dtype=torch.int16).cuda()
  assert ops.range_encode(data, cdf, 5) == oracle.best().range_encode(data.cpu().numpy(), cdf.cpu().numpy(), 5)
  with pytest.raises(ops.InvalidArgumentError, match="one more axis"):
    ops.range_encode(data, cdf.reshape(-1), 5)
  with pytest.raises(ops.InvalidArgumentError, match="Cannot broadcast"):
    ops.range_encode(data, torch.cat([cdf, cdf]), 5)
  with pytest.raises(ops.InvalidArgumentError, match="value not in"):
    ops.range_encode(torch.tensor([0, 3], dtype=torch.int16).cuda(), cdf, 5)
  with pytest.raises(ops.InvalidArgumentError, match="cdf\\[0\\]=1"):
    ops.range_encode(data, torch.tensor([[1, 16, 18, 32]], dtype=torch.int32).cuda(), 5)
  with pytest.raises(ops.InvalidArgumentError, match="cdf\\[\\^1\\]=31"):
    ops.range_encode(data, torch.tensor([[0, 16, 18, 31]], dtype=torch.int32).cuda(), 5)
  with pytest.raises(ops.InvalidArgumentError, match="monotonic"):
    ops.range_encode(data, torch.tensor([[0, 18, 16, 32]], dtype=torch.int32).cuda(), 5)
  with pytest.raises(ops.InvalidArgumentError, match="precision"):
    ops.range_encode(data, cdf, 17)


# ---- PmfToQuantizedCdf ----
PMF_CASES = [(32, 10, 0.85), (100, 7, 1.0), (257, 12, 1.3), (1500, 12, 1.0), (2, 1, 1.0), (7, 16, 0.2)]


def pmf_rows(n, scale):
  rng = np.random.default_rng(n)
  pmf = rng.random((5, n)).astype(np.float32)
  pmf[1] = pmf[1]**8           # peaky
  pmf[2, n // 2:] = 0          # half-zero row (pmf_to_cdf_kernels_test.cc:123-143)
  return (pmf / pmf.sum(-1, keepdims=True) * scale).astype(np.float32)


@pytest.mark.parametrize("n,precision,scale", PMF_CASES)
def test_pmf_to_cdf_matches_oracle(ops, n, precision, scale):
  pmf = pmf_rows(n, scale)
  got = ops.pmf_to_quantized_cdf(torch.from_numpy(pmf).cuda(), precision).cpu().numpy()
  assert got.shape == (5, n + 1)
  assert (got[:, 0] == 0).all() and (got[:, -1] == 1 << precision).all()
  assert (np.diff(got, axis=-1) >= 1).all()
  # The C port breaks ties like the kernel (lowest index, FIFO): always identical.
  assert np.array_equal(got, oracle.port().pmf_to_cdf(pmf, precision))
  # The compiled reference flavour uses std::sort: identical unless exact ties decide.
  ref = golden_util.load_reference_outputs()[f"pmf_cdf_{n}_{precision}"]
  for r in (0, 1, 3, 4):   # random rows: ties have probability ~0
    assert np.array_equal(got[r], ref[r])


def test_pmf_to_cdf_errors(ops):
  with pytest.raises(ops.InvalidArgumentError, match="non-finite or negative"):
    ops.pmf_to_quantized_cdf(torch.tensor([[0.5, float("nan"), 0.5]]).cuda(), 8)
  with pytest.raises(ops.InvalidArgumentError, match="non-finite or negative"):
    ops.pmf_to_quantized_cdf(torch.tensor([[0.5, -0.1, 0.6]]).cuda(), 8)
  with pytest.raises(ops.InvalidArgumentError, match="at least 2"):
    ops.pmf_to_quantized_cdf(torch.tensor([[1.0]]).cuda(), 8)
  with pytest.raises(ops.InvalidArgumentError, match="precision"):
    ops.pmf_to_quantized_cdf(torch.tensor([[0.5, 0.5]]).cuda(), 0)
