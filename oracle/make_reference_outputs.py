"""Generates tests/golden/reference_outputs.npz from the COMPILED REFERENCE (oracle/_ref, built by `make -C oracle ref`
where the reference tree exists): its outputs on the seeded inputs of the tests that compare the C port and the CUDA
kernels against it, so that those comparisons run wherever the repository does.
    python oracle/make_reference_outputs.py
Inputs come from the test modules themselves; every stored string was decoded back by the reference here.  The
run-length codes are stored as SHA-256 digests (the codes themselves would be most of the file)."""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import golden_util  # noqa: E402
import oracle  # noqa: E402
import test_baseline_configs_gpu  # noqa: E402
import test_misc_gpu  # noqa: E402
import test_oracle_pin as pin  # noqa: E402


def _flat(strings):
  return np.asarray([len(s) for s in strings], np.int64), np.frombuffer(b"".join(strings) + b"\0", np.uint8)[:-1]


def main():
  R = oracle.ref()
  out = {}
  # range coder fuzz: raw triples and multi-stream jobs
  triples, jobs = pin.range_coder_fuzz_cases()
  out["trip_len"], out["trip_bytes"] = _flat([R.encode_triples(lo, hi, p) for lo, hi, p in triples])
  streams = []
  for lookup, val, index in jobs:
    s = R.encode(lookup, val, index, threads=2)
    back, ok = R.decode(lookup, s, val.shape[1], index, threads=2)
    assert np.array_equal(back, val) and ok.all()
    streams += s
  out["streams_len"], out["streams_bytes"] = _flat(streams)
  # stochastic rounding with libstdc++'s seed_seq
  rng = np.random.default_rng(0)
  out["stochastic_round"] = np.stack([R.stochastic_round(x, 0.75, seed) for seed, x in pin.stochastic_round_cases(rng)])
  # run-length bit coder fuzz, with the outcome of decoding damaged codes
  codes, damaged = [], []
  big = np.iinfo(np.int32)
  for rl, mg, nz, _, d in pin.run_length_fuzz_cases():
    code = R.run_length_encode(d, rl, mg, nz)
    want = np.where(d == big.min, big.min + 1, d) if mg < 0 else d
    assert np.array_equal(R.run_length_decode(code, d.shape, rl, mg, nz), want)
    codes.append(code)
    damaged.append([pin.decode_outcome(R, c, shape, rl, mg, nz) for c, shape in pin.damaged_codes(code, d.size)])
  out["rl_code_sha256"] = np.asarray([hashlib.sha256(c).hexdigest() for c in codes])
  out["rl_damaged"] = np.asarray(damaged, dtype=str)
  # long Rice codes: the port's strings, which the reference's reader decodes
  d = pin.long_rice_data()
  long_codes = []
  for rl, mg in pin.LONG_RICE_CONFIGS:
    code = oracle.port().run_length_encode(d, rl, mg, False)
    assert np.array_equal(R.run_length_decode(code, d.shape, rl, mg, False), d)
    long_codes.append(code)
  out["long_rice_len"], out["long_rice_bytes"] = _flat(long_codes)
  # PmfToQuantizedCdf (std::sort tie order)
  for n, precision, scale in test_misc_gpu.PMF_CASES:
    out[f"pmf_cdf_{n}_{precision}"] = R.pmf_to_cdf(test_misc_gpu.pmf_rows(n, scale), precision)
  for i, pmf in enumerate(test_baseline_configs_gpu.tie_row_pmfs()):
    out[f"tie_row_cdf_{i}"] = R.pmf_to_cdf(pmf, 12)
  np.savez_compressed(golden_util.REFERENCE_OUTPUTS_PATH, **out)
  print("wrote", golden_util.REFERENCE_OUTPUTS_PATH, os.path.getsize(golden_util.REFERENCE_OUTPUTS_PATH), "bytes")


if __name__ == "__main__":
  main()
