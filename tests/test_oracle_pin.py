"""CPU: pins the oracle.  The C port must reproduce (a) the golden vectors generated from the compiled
reference, (b) the compiled reference's outputs on seeded fuzz (tests/golden/reference_outputs.npz, written by
oracle/make_reference_outputs.py from the inputs generated here)."""
import hashlib

import numpy as np
import pytest

import golden_util
import oracle
import util

FLAVOURS = ["port"] + (["ref"] if oracle.have_ref() else [])


def _o(name):
  return oracle.port() if name == "port" else oracle.ref()


@pytest.mark.parametrize("flavour", FLAVOURS)
def test_golden_vectors(flavour):
  O, g = _o(flavour), golden_util.load()
  assert O.range_encode(g["lit_data"], g["lit_cdf"], 5) == bytes(g["lit_bytes"])
  assert np.array_equal(O.range_decode(bytes(g["lit_bytes"]), g["lit_data"].shape, g["lit_cdf"], 5), g["lit_data"])
  at = 0
  want = golden_util.split(g["trip_bytes"], g["trip_len"])
  for n, w in zip(g["trip_n"], want):
    sl = slice(at, at + int(n))
    assert O.encode_triples(g["trip_lo"][sl], g["trip_hi"][sl], g["trip_p"][sl]) == w
    at += int(n)
  for mode in ("chan", "index"):
    idx = g.get(f"{mode}_index")
    want = golden_util.split(g[f"{mode}_bytes"], g[f"{mode}_len"])
    assert O.encode(g["ms_lookup"], g[f"{mode}_value"], idx) == want
    dec, ok = O.decode(g["ms_lookup"], want, g[f"{mode}_value"].shape[1], idx)
    assert np.array_equal(dec, g[f"{mode}_value"]) and ok.all()
  assert O.range_encode(g["leg_data"], g["leg_cdf"], 13) == bytes(g["leg_bytes"])
  assert np.array_equal(O.range_decode(bytes(g["leg_bytes"]), g["leg_data"].shape, g["leg_cdf"], 13), g["leg_data"])
  assert np.array_equal(O.pmf_to_cdf(g["pmf"], 10), g["pmf_cdf"])


def range_coder_fuzz_cases():
  """Seeded inputs of the port-vs-reference fuzz: 400 raw (lower, upper, precision) sequences and 60 multi-stream
  jobs (lookup, value, index)."""
  rng = np.random.default_rng(77)
  triples, jobs = [], []
  for _ in range(400):
    n = int(rng.integers(0, 150))
    prec = rng.integers(1, 17, size=n).astype(np.int32)
    tot = (1 << prec.astype(np.int64))
    lo = (rng.random(n) * tot).astype(np.int64)
    hi = lo + 1 + (rng.random(n) * (tot - lo - 1)).astype(np.int64)
    hug = rng.random(n) < 0.3
    hi[hug] = tot[hug]
    lo[hug] = tot[hug] - 1 - (rng.random(int(hug.sum())) * np.minimum(tot[hug] - 1, 3)).astype(np.int64)
    triples.append((lo, hi, prec))
  for t in range(60):
    nrows, S, N = int(rng.integers(1, 6)), int(rng.integers(1, 4)), int(rng.integers(0, 200))
    precs = [int(rng.integers(5, 17)) for _ in range(nrows)]
    cdfs = [util.random_cdf(rng, int(rng.integers(2, min(40, 1 << p) + 1)), p, peaky=3) for p in precs]
    ovf = [bool(rng.integers(0, 2)) for _ in range(nrows)]
    lookup = util.make_lookup_2d(cdfs, precs, ovf) if t % 2 else util.make_lookup_1d(cdfs, precs, ovf)
    index = rng.integers(0, nrows, size=(S, N)).astype(np.int32) if t % 3 == 0 else None
    rows = index if index is not None else np.broadcast_to(np.arange(N) % nrows, (S, N))
    nb = np.asarray([len(c) - 1 for c in cdfs])[rows]
    isov = np.asarray(ovf)[rows]
    val = (rng.random((S, N)) * np.where(isov, np.maximum(nb - 1, 1), nb)).astype(np.int32)
    wild = isov & (rng.random((S, N)) < 0.2)
    val[wild] = rng.integers(-300, 300, size=int(wild.sum()))
    jobs.append((lookup, val, index))
  return triples, jobs


def test_port_equals_compiled_reference_fuzz():
  """Same bytes as the compiled reference on every fuzz input; the generator checked that the reference decodes
  each of its strings back to the input."""
  P, g = oracle.port(), golden_util.load_reference_outputs()
  triples, jobs = range_coder_fuzz_cases()
  for (lo, hi, prec), want in zip(triples, golden_util.split(g["trip_bytes"], g["trip_len"]), strict=True):
    assert P.encode_triples(lo, hi, prec) == want
  want = golden_util.split(g["streams_bytes"], g["streams_len"])
  assert len(want) == sum(val.shape[0] for _, val, _ in jobs)
  at = 0
  for lookup, val, index in jobs:
    S, N = val.shape
    a = P.encode(lookup, val, index)
    assert a == want[at:at + S]
    at += S
    da, oka = P.decode(lookup, a, N, index)
    assert np.array_equal(da, val) and oka.all()


def test_decoder_sanity_flag_semantics():
  """RangeDecoder::Finalize (range_coder.h:144-169): unread bytes -> False; exact consumption -> True."""
  O = oracle.port()
  rng = np.random.default_rng(5)
  cdf = util.random_cdf(rng, 25, 12)
  lookup = util.make_lookup_1d([cdf], [12], [False])
  val = util.sample_symbols(rng, cdf, 900).reshape(3, 300)
  s = O.encode(lookup, val)
  _, ok = O.decode(lookup, s, 300)
  assert ok.all()
  _, ok = O.decode(lookup, s, 10)
  assert not ok.any()
  _, ok = O.decode(lookup, [x + b"\x07\x07\x07\x07" for x in s], 300)
  assert not ok.any()


def test_lookup_grammar_errors():
  """ScanCDF / IndexCDFMatrix error classes (range_coder_kernels.cc:110-164)."""
  O = oracle.port()
  for bad, msg in (([4, 1, 16], "start with 0"), ([4, 0, 3, 2, 16], "monotonically"), ([4, 0, 3], "end with"),
                   ([17, 0, 4], "precision"), ([4, 0], "prematurely")):
    with pytest.raises(oracle.OracleError, match=msg):
      O.encoder(np.asarray(bad, np.int32), 1)
  with pytest.raises(oracle.OracleError, match="end with"):
    O.encoder(np.asarray([[4, 0, 16, 16, 3]], np.int32), 1)  # 2-D row not filled with padding


def test_pmf_to_cdf_invariants_and_tie_rule():
  """pmf_to_cdf_kernels_test.cc:70-143 invariants; symmetric rows (exact ties) keep the invariants and the
  port resolves ties by lowest bin index."""
  O = oracle.port()
  rng = np.random.default_rng(9)
  for n, p, scale in ((32, 10, 0.85), (100, 7, 1.0), (41, 12, 1.15)):
    pmf = rng.random((3, n)).astype(np.float32)
    pmf[1, n // 2:] = 0
    k = np.arange(n) - (n - 1) / 2
    pmf[2] = np.exp(-0.5 * (k / (n / 8))**2)  # symmetric -> exact ties
    pmf = (pmf / pmf.sum(-1, keepdims=True) * scale).astype(np.float32)
    cdf = O.pmf_to_cdf(pmf, p)
    assert (cdf[:, 0] == 0).all() and (cdf[:, -1] == 1 << p).all() and (np.diff(cdf, axis=-1) >= 1).all()
  with pytest.raises(oracle.OracleError):
    O.pmf_to_cdf(np.asarray([[0.5, np.nan]], np.float32), 8)


STOCHASTIC_ROUND_SEEDS = ([1], [123, 456], [5] * 9, [-7, 2**31 - 1, 0, 3, 4, 5, 6, 7, 8, 9, 10])


def stochastic_round_cases(rng):
  """(seed, inputs) pairs of the port-vs-reference comparison, drawn from `rng`."""
  for seed in STOCHASTIC_ROUND_SEEDS:
    yield seed, rng.uniform(-100, 100, 20000).astype(np.float32)


def test_stochastic_round_port_equals_reference_flavour():
  """quantization_kernels.cc:48-95: the C restatement of std::seed_seq + xoshiro256+ against libstdc++'s own
  seed_seq driving the same loop (oracle/ref/ref_driver.cc; its outputs are stored), and the reference's invariants
  (python/ops/quantization_ops_test.py:28-83) on the oracle itself."""
  P, g = oracle.port(), golden_util.load_reference_outputs()
  rng = np.random.default_rng(0)
  for (seed, x), b in zip(stochastic_round_cases(rng), g["stochastic_round"], strict=True):
    a = P.stochastic_round(x, 0.75, seed)
    assert np.array_equal(a, b)
    assert np.all(np.abs(a * np.float32(0.75) - x) <= 0.75 + 1e-4)
  ints = rng.integers(-100, 100, 100).astype(np.float32)
  assert np.array_equal(P.stochastic_round(ints * np.float32(0.75), 0.75, [3]), ints.astype(np.int32))
  rep = np.broadcast_to(rng.uniform(-100, 100, 20).astype(np.float32), (20000, 20))
  assert np.abs(P.stochastic_round(rep, 1.0, [9]).mean(0) - rep[0]).max() < 3e-2


def _runs(mask):
  """Lengths of the maximal runs of True in a boolean vector."""
  edges = np.flatnonzero(np.diff(np.concatenate(([0], mask.astype(np.int8), [0]))))
  return edges[1::2] - edges[0::2]


def _inside_the_reference_writer(d, rl, mg, nz):
  """Keeps every Rice-coded quantity's unary part below 57 zeros (see the fuzz test below for why)."""
  d = d.copy()
  if mg >= 0:
    d = np.clip(d, -(56 << mg), 56 << mg).astype(np.int32)
  if rl >= 0:
    step = 56 << rl
    d[step - 1::step] = np.where(d[step - 1::step] == 0, 1, d[step - 1::step])
    if nz:
      d[step // 2::step] = 0
      assert _runs(d != 0).max(initial=0) <= step
    assert _runs(d == 0).max(initial=0) <= step
  return d


@pytest.mark.parametrize("flavour", FLAVOURS)
def test_run_length_oracles_reproduce_the_reference_literal(flavour):
  """cc/kernels/run_length_kernels_test.cc:272-305 holds the one literal bit string of the run-length ops:
  [-6, 3, 0, 0] <-> {0b11010001, 0b01101101} (gamma / gamma / zeros only); plus round trips over every code flavour."""
  P = _o(flavour)
  assert P.run_length_encode([-6, 3, 0, 0]) == bytes([0b11010001, 0b01101101])
  assert P.run_length_decode(bytes([0b11010001, 0b01101101]), (4,)).tolist() == [-6, 3, 0, 0]
  rng = np.random.default_rng(1)
  for rl, mg, nz in ((-1, -1, False), (-1, -1, True), (2, 3, True), (0, 0, False), (5, -1, False), (-1, 4, True)):
    for density in (0.02, 0.5, 1.0):
      d = (rng.integers(-300, 300, 5000) * (rng.random(5000) < density)).astype(np.int32)
      d = _inside_the_reference_writer(d, rl, mg, nz)
      code = P.run_length_encode(d, rl, mg, nz)
      assert np.array_equal(P.run_length_decode(code, d.shape, rl, mg, nz), d)
  with pytest.raises(oracle.OracleError, match="Out of bits"):
    P.run_length_decode(b"\x01", (9,))


def run_length_fuzz_cases():
  """Seeded inputs of the port-vs-reference bit coder fuzz: (rl, mg, nz, trial, data)."""
  rng = np.random.default_rng(11)
  big = np.iinfo(np.int32)
  for rl, mg, nz in ((-1, -1, False), (-1, -1, True), (0, 0, False), (2, 3, True), (5, -1, False), (-1, 4, True),
                     (3, 0, True), (7, 12, False)):
    for trial in range(12):
      n = int(rng.integers(1, 3000))
      mag = int(rng.choice([2, 40, 5000, 2**20]))
      d = (rng.integers(-mag, mag + 1, n) * (rng.random(n) < rng.choice([0.0, 0.03, 0.5, 1.0]))).astype(np.int32)
      d = _inside_the_reference_writer(d, rl, mg, nz)
      if trial == 3 and mg < 0:        # the gamma magnitude code clamps INT32_MIN to the closest value (:84-87)
        d[rng.integers(0, n)] = big.min
        d[rng.integers(0, n)] = big.max
      yield rl, mg, nz, trial, d


def damaged_codes(code, n):
  """A truncated code, and the full code read with too large and too small a tensor."""
  return ((code[:len(code) // 2], (n,)), (code, (n + 5,)), (code, (max(n - 3, 1),)))


def decode_outcome(O, code, shape, rl, mg, nz):
  """The error message of a decode, or a digest of the tensor it decoded."""
  try:
    return "sha256:" + hashlib.sha256(O.run_length_decode(code, shape, rl, mg, nz).astype(np.int32).tobytes()).hexdigest()
  except oracle.OracleError as e:
    return str(e)


def test_run_length_port_equals_the_compiled_bit_coder_fuzz():
  """The C port's own bit packing against the reference's BitWriter / BitReader (cc/lib/bit_coder.cc compiled in
  place; only the op loops of run_length_kernels.cc are restated around it; its outputs are stored): same bytes, same
  decoded tensors, same error classes on truncated and over-long codes, over every code flavour, densities from
  all-zero to dense, magnitudes up to the int32 limits.

  Inputs are kept where the reference is defined: `BitWriter::WriteRice` emits a unary part of 57 zeros or more in
  chunks of up to 57 (bit_coder.cc:88-92), and a 57-bit chunk that lands on bit offset 7 makes `WriteBits` shift its
  64-bit buffer by 64 (bit_coder.cc:60-68, undefined; on x86 the seven old bits are written twice) -- the reference
  then cannot decode its own string.  The port and the CUDA coder write the intended code there (next test)."""
  P, g = oracle.port(), golden_util.load_reference_outputs()
  big = np.iinfo(np.int32)
  for (rl, mg, nz, trial, d), ref_code, ref_outcomes in zip(run_length_fuzz_cases(), g["rl_code_sha256"],
                                                             g["rl_damaged"], strict=True):
    code = P.run_length_encode(d, rl, mg, nz)
    assert hashlib.sha256(code).hexdigest() == ref_code, (rl, mg, nz, trial)
    want = np.where(d == big.min, big.min + 1, d) if mg < 0 else d
    assert np.array_equal(P.run_length_decode(code, d.shape, rl, mg, nz), want)
    # damaged codes: the port fails in the reference's class or decodes the reference's tensor
    for (damaged, shape), ref_outcome in zip(damaged_codes(code, d.size), ref_outcomes, strict=True):
      assert decode_outcome(P, damaged, shape, rl, mg, nz) == ref_outcome, (rl, mg, nz, trial)


LONG_RICE_CONFIGS = ((0, 0), (1, 2), (0, -1))


def long_rice_data():
  d = np.zeros(5000, np.int32)
  d[[3, 700, 701, 4999]] = [9, -300, 1, 77]
  return d


def test_run_length_port_writes_long_rice_codes_as_specified():
  """Where the reference's writer is undefined (unary parts longer than 57 zeros, see above) the port follows the
  code's definition -- q zeros, a one, k low bits -- and writes the strings that the reference's own READER, which has
  no such limit, was seen to decode (stored beside the reference's outputs)."""
  P, g = oracle.port(), golden_util.load_reference_outputs()
  d = long_rice_data()
  read_by_ref = golden_util.split(g["long_rice_bytes"], g["long_rice_len"])
  for (rl, mg), want in zip(LONG_RICE_CONFIGS, read_by_ref, strict=True):
    code = P.run_length_encode(d, rl, mg, False)
    assert np.array_equal(P.run_length_decode(code, d.shape, rl, mg, False), d)
    assert code == want
  # by hand: zeros-only run of 3 then 9 with Rice(0) magnitudes: "0001" run, sign 1, 8 zeros + "1"
  code = P.run_length_encode(np.asarray([0, 0, 0, 9], np.int32), 0, 0, False)
  bits = "".join(format(b, "08b")[::-1] for b in code)       # LSB-first packing (bit_coder.cc:60)
  assert bits.startswith("0001" + "1" + "000000001")


@pytest.mark.parametrize("flavour", FLAVOURS)
def test_escape_payloads_the_reference_cannot_finish_are_refused(flavour):
  """OverflowEncode's width loop `while (gamma >= (1 << n))` (range_coder_kernels.cc:310-315, "TODO Clamp gamma")
  never ends once the payload reaches 2^30.  The checker refuses such a symbol instead of hanging (bench.py found
  this through an infinite synthetic latent); the largest payloads below the limit still round-trip."""
  O = _o(flavour)
  lookup = np.asarray([-4, 0, 5, 11, 16], np.int32)  # overflow row, escape symbol 2: payload = v - 1 for v >= 2
  fine = np.asarray([[0, 1, 1 << 30, -((1 << 30) - 1), 7, -3]], np.int32)
  s = O.encode(lookup, fine)
  back, ok = O.decode(lookup, s, fine.shape[1])
  assert np.array_equal(back, fine) and ok.all()
  for v in ((1 << 30) + 1, -(1 << 30), np.iinfo(np.int32).min, np.iinfo(np.int32).max):
    with pytest.raises(oracle.OracleError, match="Elias-gamma payload"):
      O.encode(lookup, np.asarray([[0, v, 0]], np.int32))


def test_bench_latents_are_finite_on_every_rank():
  """bench.synth_latents: rand() == 0 used to give log1p(-1) = -inf, i.e. a latent that quantises to INT32_MIN;
  rank 1's first batch had one, and the per-rank parity check then waited for ever inside the oracle."""
  import torch
  import bench
  for rank in (0, 1, 7):
    _, ys = bench.synth_latents(rank, 2, batch=64)
    assert all(bool(torch.isfinite(y).all()) and float(y.abs().max()) < 8.0 * 17.0 + 1e-3 for y in ys)
  _, full = bench.synth_latents(1, 1)   # the batch that hung the 2-GPU run
  assert bool(torch.isfinite(full[0]).all())


@pytest.mark.parametrize("flavour", FLAVOURS)
def test_run_length_golden_vectors(flavour):
  """tests/golden/run_length_golden.npz (oracle/make_run_length_golden.py: strings written by the reference's own
  BitWriter): every oracle flavour reproduces the bytes and decodes them."""
  import os
  g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "run_length_golden.npz"))
  O = _o(flavour)
  at_d = at_c = 0
  for (rl, mg, nz), nd, nc in zip(g["params"], g["data_len"], g["code_len"]):
    d = g["data"][at_d:at_d + nd]
    code = bytes(g["code"][at_c:at_c + nc])
    at_d, at_c = at_d + nd, at_c + nc
    assert O.run_length_encode(d, int(rl), int(mg), bool(nz)) == code
    assert np.array_equal(O.run_length_decode(code, d.shape, int(rl), int(mg), bool(nz)), d)
  assert bytes(g["code"][:2]) == bytes([0b11010001, 0b01101101])   # the reference test's literal
