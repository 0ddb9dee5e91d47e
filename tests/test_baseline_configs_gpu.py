"""GPU parity AT THE BASELINE CONFIG SIZES (BASELINE.json configs[0..2], SURVEY.md 8(d)): the CUDA path's bytes against
the compiled-reference oracle, and both cross-decodes, on the full cfg1 / cfg2 / cfg3 workloads that bench.py times.

Reference behaviour: continuous_batched.py:347-422, continuous_indexed.py:354-417 (model methods),
cc/kernels/range_coder_kernels.cc:191-322,360-471 (stream loops), cc/kernels/range_coding_kernels_test.cc:246-322
(legacy op shapes)."""
import os

import numpy as np
import pytest
import torch

import bench
import golden_util
import oracle

pytestmark = pytest.mark.gpu

THREADS = os.cpu_count() or 1


def _symbols(em, y, index=None, loc=None):
  q = getattr(em, "quantization_offset", None) if index is None else None
  b = y.cpu()
  if q is not None:
    b = b - q.cpu()
  if loc is not None:
    b = b - loc.cpu()
  coff = em.cdf_offset.cpu()
  sym = torch.round(b).to(torch.int32) - (coff if index is None else coff[index.long().cpu()])
  return sym.reshape(y.shape[0], -1).numpy()


@pytest.mark.parametrize("prior", ["laplace", "deep"])
def test_cfg2_full_size_bytes_equal_oracle(prior):
  """256 streams x 32 768 symbols, 128 channel tables (the bench's NoisyLaplace tables and the models' own
  NoisyDeepFactorized), fused and literal op sequences, both cross-decodes."""
  dev = torch.device("cuda", 0)
  scales, ys = bench.synth_latents(0, 1)
  em = bench.build_model(scales, dev, prior)
  y = ys[0] if prior == "laplace" else ys[0] * 2.5   # the default deep-factorised prior is ~ +-30 wide
  assert y.shape == (256, 16, 16, 128)
  O = oracle.best()
  lookup = em.cdf.cpu().numpy()
  value = _symbols(em, y)
  want = O.encode(lookup, value, None, THREADS)
  got = em.compress(y.to(dev))
  assert got.shape == (256,)
  assert got.tolist() == want
  assert em.compress(y.to(dev), fused=False).tolist() == want
  # the oracle decodes the GPU's strings; the GPU decodes the oracle's (fused and literal)
  back, ok = O.decode(lookup, got.tolist(), value.shape[1], None, THREADS)
  assert np.array_equal(back, value) and ok.all()
  yq = em.quantize(y.to(dev))
  assert torch.equal(em.decompress(want, (16, 16)), yq)
  assert torch.equal(em.decompress(want, (16, 16), fused=False), yq)
  # escapes really occur at this size (tail_mass 2^-8): the Elias-gamma path is part of the check
  nb = np.diff(np.flatnonzero(np.r_[lookup < 0, True])) - 3 if lookup.ndim == 1 else None
  assert (value < 0).any() or (nb is not None and (value >= np.tile(nb, value.shape[1] // len(nb))).any())


def test_cfg3_full_size_bytes_equal_oracle():
  """bmshj2018 two-level: y[128,16,16,192] in index mode over all 64 NoisyNormal tables (sigma up to 256, > 1000 bins),
  with loc; z[128,4,4,192] in channel mode.  Encode and decode, both levels, against the oracle."""
  dev = torch.device("cuda", 0)
  w = bench.cfg3_workload(dev)
  em_y, em_z, y, idx, loc, z = (w[k] for k in ("em_y", "em_z", "y", "idx", "loc", "z"))
  O = oracle.best()
  flat = torch.clamp(idx, 0, 63).to(torch.int32)
  assert int(flat.min()) == 0 and int(flat.max()) == 63          # every table, including sigma = 256
  index = flat.reshape(128, -1).cpu().numpy()
  lookup_y = em_y.cdf.cpu().numpy()
  value = _symbols(em_y, y, index=flat, loc=loc)
  want = O.encode(lookup_y, value, index, THREADS)
  got = em_y.compress(y, idx, loc=loc)
  assert got.tolist() == want
  assert em_y.compress(y, idx, loc=loc, fused=False).tolist() == want
  back, ok = O.decode(lookup_y, got.tolist(), value.shape[1], index, THREADS)
  assert np.array_equal(back, value) and ok.all()
  yq = em_y.quantize(y, loc)
  assert torch.equal(em_y.decompress(want, idx, loc=loc), yq)
  assert torch.equal(em_y.decompress(want, idx, loc=loc, fused=False), yq)
  # z: channel mode, 192 tables
  lookup_z = em_z.cdf.cpu().numpy()
  vz = _symbols(em_z, z)
  want_z = O.encode(lookup_z, vz, None, THREADS)
  got_z = em_z.compress(z)
  assert got_z.tolist() == want_z
  assert torch.equal(em_z.decompress(want_z, (4, 4)), em_z.quantize(z))


@pytest.mark.parametrize("per_channel", [False, True])
def test_cfg1_legacy_op_exactly_as_stated(per_channel):
  """data[1,16,16,128] int16, cdf[1,1,1,1,65] / cdf[1,1,1,128,65], precision 14: RangeEncode bytes == the oracle's,
  oracle-decode(GPU bytes) == symbols, GPU-decode(oracle bytes) == symbols."""
  from compression_b200 import gen_ops
  data, cdf, precision = bench.cfg1_workload(per_channel)
  assert data.shape == (1, 16, 16, 128) and cdf.shape == ((1, 1, 1, 128, 65) if per_channel else (1, 1, 1, 1, 65))
  O = oracle.best()
  want = O.range_encode(data, cdf, precision)
  got = gen_ops.range_encode(torch.from_numpy(data).cuda(), torch.from_numpy(cdf).cuda(), precision)
  assert got == want
  assert np.array_equal(O.range_decode(got, data.shape, cdf, precision), data)
  dec = gen_ops.range_decode(want, list(data.shape), torch.from_numpy(cdf).cuda(), precision)
  assert dec.dtype == torch.int16 and np.array_equal(dec.cpu().numpy(), data)


def tie_row_pmfs():
  """One symmetric discretised-normal PMF row for every 7th of the 64 cfg3 scales."""
  from scipy.stats import norm
  sig = np.exp(np.log(.11) + np.arange(64) * (np.log(256.) - np.log(.11)) / 63)
  pmfs = []
  for s in sig[::7]:
    half = int(np.ceil(s * 2.8)) + 1
    k = np.arange(-half, half + 1, dtype=np.float64)
    pmfs.append((norm.cdf((k + .5) / s) - norm.cdf((k - .5) / s)).astype(np.float32)[None])
  return pmfs


def test_pmf_to_cdf_tie_rows_distance_to_the_compiled_reference():
  """a-7 on tie rows (every symmetric NoisyNormal table of cfg3): the kernel equals the C port (lowest-index tie
  break); against the compiled-reference flavour (libstdc++ std::sort order; its tables are stored) the tables may
  differ only by moving single counts between bins of EQUAL mass -- recorded here: identical bin-count multiset,
  |difference| <= 1 per bin, and a coding-cost difference of exactly zero under the table's own PMF."""
  from compression_b200 import gen_ops
  refs = golden_util.load_reference_outputs()
  worst = 0
  for i, pmf in enumerate(tie_row_pmfs()):
    got = gen_ops.pmf_to_quantized_cdf(torch.from_numpy(pmf).cuda(), 12).cpu().numpy()
    assert np.array_equal(got, oracle.port().pmf_to_cdf(pmf, 12))
    ref = refs[f"tie_row_cdf_{i}"]
    a, b = np.diff(got[0]), np.diff(ref[0])
    assert sorted(a) == sorted(b)
    assert np.abs(a - b).max() <= 1
    moved = np.flatnonzero(a != b)
    # counts only move between bins whose float masses are equal (mirror-image bins of the symmetric PMF)
    assert np.array_equal(np.sort(pmf[0][moved]), np.sort(pmf[0][moved][::-1]))
    assert np.allclose(np.sort(pmf[0][moved])[::2], np.sort(pmf[0][moved])[1::2]) if len(moved) % 2 == 0 else True
    worst = max(worst, len(moved))
  print("bins that differ from the compiled-reference flavour on symmetric tables (max over rows):", worst)
