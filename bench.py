"""bench.py -- headline benchmark of the B200-native tensorflow/compression hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--no-extras] [--dump-outputs DIR]
    (N > 1: launched by `python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...`)

Workload (BASELINE.json configs[1], "cfg2"): bls2017 compress path at batch 256, 256x256x3 images,
num_filters=128  ->  latents y [256,16,16,128] fp32 (256 code streams x 32768 symbols, 128 channel
tables, precision 12, overflow/Elias-gamma escape enabled).  One STEP = one pass of the entropy-bottleneck
hot path over one batch: quantise (y - offset -> rint -> - cdf_offset), range-encode every stream,
finalize and pack the strings (ContinuousBatchedEntropyModel.compress).  The decode path, the GDN layers,
cfg3 (bmshj2018 two-level) and the image -> strings model path are measured in the same run and reported in
the `decode` / `gdn` / `cfg3_bmshj2018` / `model_path` objects of the JSON line (extras, rank 0, N = 1).

`value`   = symbols / s with y resident in HBM (whole job, all ranks), EXACTLY K steps, CUDA events.
`e2e`     = the same metric through the public API with HOST buffers: pinned-host y -> H2D -> compress ->
            D2H of the packed strings + offsets, every step; the K-step region is repeated 7 times and the
            median is reported (min / max beside it).
`--impl reference` = the reference's own CPU range coder (oracle/_ref: cc/lib/range_coder.cc compiled in
            place, driven by the restated op loops on a persistent pool of all host threads), same symbols
            and tables (tests/golden/cfg2_tables.npz, written by tools/make_cfg_fixtures.py from the product's
            table builder); this arm never imports compression_b200.
Parity: outside the timed region every rank checks its first batch against the oracle, byte for byte, and
cross-decodes it (`parity_checked`).
`--dump-outputs DIR` = after the timed steps, rank 0 writes the strings its last timed step produced (both arms) as
            DIR/strings_bytes.npy (float32, one element per byte, all strings back to back) and
            DIR/strings_offsets.npy (float64, the S + 1 offsets delimiting them); the inputs are seeded, so two builds
            run with the same arguments can be compared output for output.

Weak scaling: every rank codes its own 256-stream batch; rank 0 builds the tables and broadcasts them
(NCCL); there is no data-path collective.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

CFG = dict(batch=256, hw=16, channels=128, precision=12, tail_mass=2**-8, n_rot=6)
METRIC = "range-code throughput (bls2017 compress path, cfg2)"
WORKLOAD = ("cfg2: bls2017 compress, y[256,16,16,128] fp32 per GPU, 256 streams x 32768 symbols, "
            "128 NoisyLaplace channel tables, precision 12, overflow on; step = quantise + range-encode + "
            "finalize/pack")
FIXTURE = os.path.join(ROOT, "tests", "golden", "cfg2_tables.npz")
E2E_REPEATS = 7


def _peaks():
  path = os.path.join(ROOT, "MEASURED_PEAKS.json")
  if os.path.exists(path):
    with open(path) as f:
      p = json.load(f)
    return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
  return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# Workloads (SURVEY.md 8(d)); shared with tests/test_baseline_configs_gpu.py
# ------------------------------------------------------------------------------------------------
def synth_latents(rank, n_rot, batch=None):
  """cfg2: y[b,h,w,c] ~ Laplace(0, s_c), s_c log-spaced 0.3..8 over channels (seed 2)."""
  import torch
  C, B, HW = CFG["channels"], batch or CFG["batch"], CFG["hw"]
  g = torch.Generator().manual_seed(2 + 1000 * rank)
  scales = torch.exp(torch.linspace(np.log(0.3), np.log(8.0), C))
  out = []
  for _ in range(n_rot):
    u = torch.rand(B, HW, HW, C, generator=g) - 0.5
    # rand() returns exactly 0 about once per 2^24 draws, i.e. u = -0.5 and log1p(-1) = -inf: an infinite latent
    # quantises to INT32_MIN, whose Elias-gamma payload the reference's width loop never finishes
    # (range_coder_kernels.cc:310-315).  Every other draw has 1 - 2|u| >= 2^-23 (log >= -15.95), so the clamp
    # touches only those draws.
    y = -scales * torch.sign(u) * torch.log1p(-2 * u.abs()).clamp_min(-17.0)
    out.append(y.contiguous())
  return scales, out


def build_model(scales, device, prior="laplace"):
  """cfg2 entropy model: ContinuousBatchedEntropyModel over per-channel NoisyLaplace priors (bench) or the
  models' own NoisyDeepFactorized(batch_shape=(128,)) (models/bls2017.py:103); both exercise the device table
  builder, tfcb_build_lookup."""
  import torch
  import compression_b200 as tfc
  if prior == "laplace":
    p = tfc.NoisyLaplace(loc=torch.zeros_like(scales), scale=scales)
  else:
    torch.manual_seed(11)
    p = tfc.NoisyDeepFactorized(batch_shape=(len(scales),))
  return tfc.ContinuousBatchedEntropyModel(p, coding_rank=3, compression=True, tail_mass=CFG["tail_mass"],
                                           range_coder_precision=CFG["precision"]).to(device)


def cfg3_workload(dev, batch=128):
  """cfg3 (bmshj2018, batch 128 of 256x256): y[128,16,16,192] coded by LocationScaleIndexedEntropyModel over
  64 NoisyNormal tables sigma = exp(log .11 + i (log 256 - log .11)/63), indexes uniform in [0, 64) as floats
  (seed 5), y ~ loc + N(0, sigma_idx); z[128,4,4,192] ~ N(0, s_c) coded by the batched model (NoisyLaplace)."""
  import torch
  import compression_b200 as tfc
  C3, num_scales, smin, smax = 192, 64, .11, 256.
  off3, fac3 = np.log(smin), (np.log(smax) - np.log(smin)) / (num_scales - 1.)
  scale_fn = lambda i: torch.exp(off3 + fac3 * i)
  em_y = tfc.LocationScaleIndexedEntropyModel(tfc.NoisyNormal, num_scales, scale_fn, coding_rank=3, compression=True)
  g = torch.Generator().manual_seed(5)
  idx = torch.rand(batch, 16, 16, C3, generator=g) * num_scales
  sig = scale_fn(torch.clamp(idx, 0, num_scales - 1).to(torch.int32).float())
  loc = torch.randn(batch, 16, 16, C3, generator=g)
  y = loc + sig * torch.randn(batch, 16, 16, C3, generator=g)
  zs = torch.exp(torch.linspace(np.log(0.5), np.log(6.0), C3))
  em_z = tfc.ContinuousBatchedEntropyModel(tfc.NoisyLaplace(loc=torch.zeros_like(zs), scale=zs), coding_rank=3,
                                           compression=True).to(dev)
  z = torch.randn(batch, 4, 4, C3, generator=g) * zs
  return dict(em_y=em_y, em_z=em_z, y=y.to(dev), idx=idx.to(dev), loc=loc.to(dev), z=z.to(dev),
              workload="bmshj2018 two-level: y[128,16,16,192] indexed NoisyNormal (64 scales up to sigma=256, "
                       "loc) + z[128,4,4,192] batched NoisyLaplace; 128 streams each")


def cfg1_workload(per_channel):
  """cfg1 exactly as SURVEY.md 8(d): one image of 32 768 int16 symbols, legacy op shapes data[1,16,16,128] with
  cdf[1,1,1,1,65] or cdf[1,1,1,128,65]; 64-bin discretised Laplace/Gaussian PMFs integerised at precision 14 by the
  oracle's PerShard; symbols drawn from the PMF (torch.manual_seed(0))."""
  import torch
  import oracle
  torch.manual_seed(0)
  rows = 128 if per_channel else 1
  k = np.arange(64) - 31.5
  pmfs = []
  for r in range(rows):
    s = 2.0 + 10.0 * r / max(rows - 1, 1)
    w = np.exp(-np.abs(k) / s) if r % 2 == 0 else np.exp(-0.5 * (k / s)**2)
    pmfs.append((w / w.sum()).astype(np.float32))
  pmf = np.stack(pmfs)
  cdf = oracle.port().pmf_to_cdf(pmf, 14)                       # [rows, 65]
  p = torch.from_numpy(np.diff(cdf, axis=-1).astype(np.float64))
  data = torch.multinomial(p / p.sum(-1, keepdim=True), 256 * (128 // rows), replacement=True)  # [rows, n]
  data = data.t().reshape(1, 16, 16, 128).to(torch.int16).numpy() if per_channel else \
      data.reshape(1, 16, 16, 128).to(torch.int16).numpy()
  cshape = (1, 1, 1, 128, 65) if per_channel else (1, 1, 1, 1, 65)
  return data, cdf.reshape(cshape).astype(np.int32), 14


def symbols_of(cdf_offset, qoff, y):
  """Host int32 symbols exactly as ContinuousBatchedEntropyModel.compress derives them
  (continuous_batched.py:375-380)."""
  import torch
  b = y if qoff is None else y - torch.as_tensor(qoff)
  sym = torch.round(b).to(torch.int32) - torch.as_tensor(cdf_offset, dtype=torch.int32)
  return sym.reshape(y.shape[0], -1).numpy()


def load_fixture():
  """cfg2 tables written once from the product's table builder (tools/make_cfg_fixtures.py)."""
  if not os.path.exists(FIXTURE):
    return None
  z = np.load(FIXTURE)
  return dict(lookup=z["lookup"], cdf_offset=z["cdf_offset"],
              qoff=(z["quantization_offset"] if z["has_qoff"] else None))


def dump_strings(out_dir, strings):
  """Writes a batch of byte strings as the arrays a caller receives: the bytes back to back and their offsets."""
  offsets = np.concatenate([[0], np.cumsum([len(s) for s in strings])]).astype(np.float64)
  raw = np.frombuffer(b"".join(strings), np.uint8).astype(np.float32)
  assert raw.nbytes + offsets.nbytes <= 64 << 20, "the dumped outputs would exceed 64 MB"
  os.makedirs(out_dir, exist_ok=True)
  np.save(os.path.join(out_dir, "strings_bytes.npy"), raw)
  np.save(os.path.join(out_dir, "strings_offsets.npy"), offsets)


def stand_in_tables(scales):
  """Only when the fixture is missing: Laplace tables of the same widths from tests/util.py."""
  sys.path.insert(0, os.path.join(ROOT, "tests"))
  import util
  cdfs = [util.laplace_cdf(2 * int(6 * s + 3) + 1, CFG["precision"], float(s)) for s in scales]
  lookup = util.make_lookup_1d(cdfs, [CFG["precision"]] * len(cdfs), [True] * len(cdfs))
  off = -np.asarray([(len(c) - 1) // 2 for c in cdfs], np.int32)
  return dict(lookup=lookup, cdf_offset=off, qoff=None)


# ------------------------------------------------------------------------------------------------
# Host placement, clocks
# ------------------------------------------------------------------------------------------------
def pin_to_gpu_numa_node(dev_index):
  """Pins the process (and the threads it spawns later) to the CPUs of the GPU's NUMA node: the H2D/D2H copies
  and the launch thread then do not cross the socket interconnect.  Best effort; returns what was done."""
  try:
    import torch
    p = torch.cuda.get_device_properties(dev_index)
    bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
    with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
      node = int(f.read())
    if node < 0:
      return {"node": node, "pinned": False}
    with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
      cpus = set()
      for part in f.read().strip().split(","):
        a, _, b = part.partition("-")
        cpus.update(range(int(a), int(b or a) + 1))
    cpus &= os.sched_getaffinity(0)
    if not cpus:
      return {"node": node, "pinned": False}
    os.sched_setaffinity(0, cpus)
    return {"node": node, "pinned": True, "cpus": len(cpus)}
  except Exception as e:  # pylint:disable=broad-except
    return {"pinned": False, "why": repr(e)[:80]}


def physical_cores():
  try:
    seen = set()
    phys = core = None
    with open("/proc/cpuinfo") as f:
      for line in f:
        if line.startswith("physical id"):
          phys = line.split(":")[1].strip()
        elif line.startswith("core id"):
          core = line.split(":")[1].strip()
        elif not line.strip():
          if phys is not None and core is not None:
            seen.add((phys, core))
          phys = core = None
    return len(seen) or (os.cpu_count() or 1)
  except Exception:  # pylint:disable=broad-except
    return os.cpu_count() or 1


class ClockSampler:
  """Samples SM clocks / throttle reasons while the timed region runs (in-process NVML, else nvidia-smi)."""
  Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
       "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

  def __init__(self, index, uuid=None):
    self.index, self.uuid, self.rows, self._stop = index, uuid, [], threading.Event()
    self._t = threading.Thread(target=self._run, daemon=True)

  def _run_nvml(self):
    import pynvml
    pynvml.nvmlInit()
    h = None
    if self.uuid:
      for u in (self.uuid, "GPU-" + self.uuid):
        try:
          h = pynvml.nvmlDeviceGetHandleByUUID(u if isinstance(u, bytes) else u.encode())
          break
        except Exception:  # pylint:disable=broad-except
          h = None
    if h is None:
      h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
    mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
    get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
    bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
    while not self._stop.is_set():
      sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
      r = int(get_reasons(h))
      self.rows.append([str(sm), str(mx)] + [("Active" if r & bits[n] else "Not Active")
                                              for n in ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")])
      self._stop.wait(0.05)

  def _run(self):
    try:
      self._run_nvml()
      return
    except Exception:  # pylint:disable=broad-except
      pass
    while not self._stop.is_set():
      try:
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
        self.rows.append([c.strip() for c in out.strip().split(",")])
      except Exception:  # pylint:disable=broad-except
        pass
      self._stop.wait(0.5)

  def __enter__(self):
    self._t.start()
    return self

  def __exit__(self, *a):
    self._stop.set()
    self._t.join(timeout=6)

  def summary(self):
    sm = [int(r[0]) for r in self.rows if len(r) >= 6 and r[0].isdigit()]
    mx = [int(r[1]) for r in self.rows if len(r) >= 6 and r[1].isdigit()]
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    reasons = sorted({n for r in self.rows if len(r) >= 6 for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
    return {"sm_mhz": int(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
            "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU legs (the only places that execute oracle/)
# ------------------------------------------------------------------------------------------------
def cpu_coder_times(value, lookup, threads, repeats=5, decode=True):
  """Median Msymbols/s of the reference CPU coder (EntropyEncodeChannel + Finalize, and CreateRangeDecoder +
  EntropyDecodeChannel + Finalize) over `repeats` runs after one warm-up; the worker pool persists."""
  import oracle
  O = oracle.best()
  S, N = value.shape
  enc_t, dec_t, strings = [], [], None
  for i in range(repeats + 1):
    enc = O.encoder(lookup, S)
    t0 = time.perf_counter()
    enc.encode(value, None, threads)
    strings = enc.finalize()
    dt = time.perf_counter() - t0
    enc.close()
    if i:
      enc_t.append(dt)
  if decode:
    for i in range(repeats + 1):
      t0 = time.perf_counter()
      dec = O.decoder(strings, lookup)
      out = dec.decode(N, None, threads)
      dec.finalize()
      dt = time.perf_counter() - t0
      dec.close()
      if i:
        dec_t.append(dt)
    assert np.array_equal(out, value)
  f = lambda ts: {"median": S * N / float(np.median(ts)) / 1e6, "min": S * N / max(ts) / 1e6,
                  "max": S * N / min(ts) / 1e6} if ts else None
  return f(enc_t), f(dec_t), O.kind


def cpu_gdn_baseline(C=192, n_pix=262144, repeats=3):
  """PyTorch-CPU fp32 GDN (abs -> matmul -> + beta -> div; SURVEY.md 8(d)) on all host threads; GB/s on the
  same algorithmic-bytes scale as the GPU numbers (8 B/element)."""
  import torch
  g = torch.Generator().manual_seed(4)
  gamma = 0.1 * torch.eye(C) + (0.02 * torch.randn(C, C, generator=g)).abs()
  beta = 1 + 0.5 * torch.rand(C, generator=g)
  x = torch.randn(n_pix, C, generator=g)
  ts = []
  for i in range(repeats + 1):
    t0 = time.perf_counter()
    y = x / (x.abs() @ gamma + beta)
    dt = time.perf_counter() - t0
    if i:
      ts.append(dt)
  del y
  gbs = 8.0 * n_pix * C / float(np.median(ts)) / 1e9
  return {"fwd_GBps": gbs, "threads": torch.get_num_threads(), "sample": f"[{n_pix},{C}] fp32, median of {repeats}"}


def warm_oracle_pool():
  """Creates the oracle's persistent workers now (unpinned, one per host thread), with a trivial job."""
  import oracle
  cores = os.cpu_count() or 1
  lookup = np.asarray([4, 0, 8, 16], np.int32)
  oracle.best().encode(lookup, np.zeros((cores, 1), np.int32), None, cores)


def sweep_threads(value, lookup, cores, reps=2):
  """Throughput of the reference CPU encoder for T = 1, 2, 4 ... host threads (best of `reps` each): boxes whose
  cgroup quota is far below their logical CPU count run SLOWER with one thread per logical CPU, so "all the host
  threads it can use" is the T that codes fastest.  Returns ({T: Msym/s}, best T)."""
  import oracle
  O = oracle.best()
  S, N = value.shape
  cand = sorted({min(cores, 1 << k) for k in range(0, 12)} | {cores})
  res = {}
  for t in cand:
    best = None
    for _ in range(reps):
      e = O.encoder(lookup, S)
      t0 = time.perf_counter()
      e.encode(value, None, t)
      e.finalize()
      dt = time.perf_counter() - t0
      e.close()
      best = dt if best is None else min(best, dt)
    res[t] = S * N / best / 1e6
  return res, max(res, key=res.get)


def run_reference(args):
  """--impl reference: rank 0 only; every step codes the full cfg2 batch on the host cores.  Never imports
  compression_b200: tables come from the committed fixture."""
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return
  import oracle
  scales, ys = synth_latents(0, 1)
  cores = os.cpu_count() or 1
  tab = load_fixture()
  tables = "tests/golden/cfg2_tables.npz (product table builder)"
  if tab is None:
    tab, tables = stand_in_tables(scales), "stand-in Laplace tables (fixture missing)"
  value = symbols_of(tab["cdf_offset"], tab["qoff"], ys[0])
  lookup = tab["lookup"]
  O = oracle.best()
  S, N = value.shape
  sweep, threads = sweep_threads(value, lookup, cores)

  def one():
    e = O.encoder(lookup, S)
    e.encode(value, None, threads)
    strings = e.finalize()
    e.close()
    return strings

  for _ in range(max(args.warmup, 1)):
    one()
  # the K-step region, repeated: the line's value is the median region
  regions = []
  for _ in range(E2E_REPEATS):
    t0 = time.perf_counter()
    for _ in range(args.steps):
      last = one()
    regions.append(time.perf_counter() - t0)
  if args.dump_outputs:
    dump_strings(args.dump_outputs, last)
  dt = float(np.median(regions))
  val = S * N * args.steps / dt / 1e6
  spread = {"min": S * N * args.steps / max(regions) / 1e6, "max": S * N * args.steps / min(regions) / 1e6,
            "repeats": len(regions)}
  sample = (f"full cfg2 batch ({S} streams x {N} int32 symbols) per step; EntropyEncodeChannel+Finalize only; "
            f"persistent pool, {threads} threads (fastest of the sweep over 1..{cores}); median of {len(regions)} regions "
            f"of {args.steps} steps")
  print(json.dumps({
      "impl": "reference", "metric": METRIC, "value": val,
      "unit": "Msymbols/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": max(args.warmup, 1),
      "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
      "dtype": "u32", "data": "synthetic",
      "config": {"workload": WORKLOAD, "tables": tables},
      "spread": spread,
      "cpu_baseline": {"value": val, "unit": "Msymbols/s", "cores": threads, "logical_cpus": cores, "kind": O.kind,
                       "sample": sample, "thread_sweep_msym_s": {str(k): round(v, 1) for k, v in sweep.items()}},
      "e2e": {"value": val, "unit": "Msymbols/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
  }))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def _time_ms(fn, reps, warm=1):
  """Median device time of one call: `reps` calls back to back with a CUDA event between consecutive calls.
  The warm-up keeps the previous result alive exactly as the timed loop does, so that the caching allocator
  already holds both output buffers (a cudaMalloc of a 0.5 - 13 GB output inside the timed region stalls the
  launch thread for milliseconds and used to be averaged into the GDN numbers)."""
  import torch
  out = None
  for _ in range(max(warm, 2)):
    out = fn()
  ev = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
  torch.cuda.synchronize()
  ev[0].record()
  for i in range(reps):
    out = fn()
    ev[i + 1].record()
  torch.cuda.synchronize()
  return float(np.median([ev[i].elapsed_time(ev[i + 1]) for i in range(reps)])), out


def parity_check(model, y_host, strings, threads):
  """One batch against the oracle: same bytes, oracle decodes ours, we decode the oracle's."""
  import torch
  import oracle
  O = oracle.best()
  lookup = model._lookup_host()
  q = model.quantization_offset
  value = symbols_of(model.cdf_offset.cpu().numpy(), None if q is None else q.cpu(), y_host)
  want = O.encode(lookup, value, None, threads)
  got = strings.tolist()
  same = got == want
  back, ok = O.decode(lookup, got, value.shape[1], None, threads)
  cross1 = bool(np.array_equal(back, value) and ok.all())
  dec = model.decompress(want, (CFG["hw"], CFG["hw"]))
  cross2 = bool(torch.equal(dec.cpu(), model.quantize(y_host)))
  return bool(same and cross1 and cross2), {"bytes_equal": bool(same), "oracle_decodes_gpu": cross1,
                                           "gpu_decodes_oracle": cross2, "oracle": O.kind}


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=200)
  ap.add_argument("--warmup", type=int, default=5)
  ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
  ap.add_argument("--no-extras", action="store_true", help="skip the decode / GDN / cfg3 / model-path / CPU side measurements")
  ap.add_argument("--dump-outputs", metavar="DIR", help="write the strings of the last timed step to DIR as .npy")
  args = ap.parse_args()
  if args.steps < 1:
    ap.error("--steps must be at least 1")
  if args.impl == "reference":
    return run_reference(args)

  import torch
  import torch.distributed as dist
  import compression_b200 as tfc
  from compression_b200 import _lib, functional, gen_ops, sharding

  rank = int(os.environ.get("RANK", "0"))
  world = int(os.environ.get("WORLD_SIZE", "1"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
  # A rank stuck outside a collective leaves the others waiting in NCCL for ever: every rank arms a watchdog
  # that prints all its Python stacks and exits non-zero instead (re-armed before each phase).
  import faulthandler
  watchdog_s = int(os.environ.get("TFCB_BENCH_WATCHDOG_S", "900"))

  def phase(name):
    faulthandler.cancel_dump_traceback_later()
    if world > 1:   # a single process has nobody to leave waiting: no limit on its side measurements
      faulthandler.dump_traceback_later(watchdog_s, exit=True)
    if os.environ.get("TFCB_BENCH_TRACE"):
      print(f"[bench rank {rank}] {name}", file=sys.stderr, flush=True)

  phase("setup")
  torch.cuda.set_device(local)
  dev = torch.device("cuda", local)
  warm_oracle_pool()                      # before pinning: the checker's workers keep the whole machine
  numa = pin_to_gpu_numa_node(local)
  if world > 1:
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    import datetime
    dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(minutes=30))

  n_rot = CFG["n_rot"]
  scales, ys_host = synth_latents(rank, n_rot)
  # rank 0 builds the tables; everyone else receives them (the only collective on the path)
  if rank == 0:
    model = build_model(scales, dev)
  else:
    model = tfc.ContinuousBatchedEntropyModel(prior_shape=(CFG["channels"],), coding_rank=3, compression=True,
                                              cdf_shapes=(1, 1), quantization_offset=True).to(dev)
  sharding.broadcast_tables(model, src=0, device=dev)

  ys = [y.to(dev) for y in ys_host]          # > L2: 6 x 33.5 MB rotate through the timed steps
  ys_pinned = [y.pin_memory() for y in ys_host]
  S = CFG["batch"]
  N = ys[0].numel() // S
  sym_per_step = S * N

  def step(i):
    return model.compress(ys[i % n_rot])

  def barrier():
    torch.cuda.synchronize()
    if world > 1:
      dist.barrier()

  def allmax(ms):
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())

  phase("warm-up")
  for i in range(max(args.warmup, 3)):
    strings = step(i)
  barrier()
  bits_per_symbol = 8.0 * strings.nbytes() / sym_per_step

  # ---- parity, outside the timed region: every rank, its own first batch, byte for byte against the oracle ----
  phase("parity")
  threads = max(1, (os.cpu_count() or 1) // world)
  ok, parity = parity_check(model, ys_host[0], model.compress(ys[0]), threads)
  flag = torch.tensor([1 if ok else 0], device=dev)
  if world > 1:
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
  parity["all_ranks"] = bool(flag.item())
  fixture = load_fixture()
  tables_match = None if fixture is None else bool(np.array_equal(fixture["lookup"], model._lookup_host()))

  # ---- the timed region: exactly K steps, CUDA events, max over ranks; returns the last step's strings too ----
  def timed_region(k):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(k):
      last = step(i)
    ev1.record()
    barrier()
    return allmax(ev0.elapsed_time(ev1)), last

  phase("timed region")
  launches0 = _lib.launch_count()
  # clocks are sampled by rank 0 only (its own GPU, in-process NVML): one sampler per rank disturbed the others
  clocks = ClockSampler(local, str(torch.cuda.get_device_properties(dev).uuid)) if rank == 0 else None
  if clocks:
    clocks.__enter__()
  elapsed_ms, last_strings = timed_region(args.steps)
  if clocks:
    clocks.__exit__()
  launches = _lib.launch_count() - launches0
  value = world * sym_per_step * args.steps / (elapsed_ms * 1e-3) / 1e6
  more = [timed_region(args.steps)[0] for _ in range(4)]   # informational spread of the same region
  vals = sorted(world * sym_per_step * args.steps / (m * 1e-3) / 1e6 for m in [elapsed_ms] + more)

  # ---- e2e: pinned host y -> H2D -> compress -> D2H(bytes, offsets), same K steps ----
  # Two staging buffers and a copy stream: the H2D copy of batch i+1 runs while batch i is encoded (compress()
  # blocks the host at its finalize, so the next copy has to be queued before it).  Every step's H2D and D2H
  # happen inside the timed region; the result (bytes + offsets) lands in pinned host memory.
  phase("e2e")
  out_cap = 2 * strings.nbytes() + 4096
  host_bytes = [torch.empty(out_cap, dtype=torch.uint8).pin_memory() for _ in range(2)]
  host_offs = [torch.empty(S + 1, dtype=torch.int64).pin_memory() for _ in range(2)]
  stages = [torch.empty_like(ys[0]) for _ in range(2)]
  copy_stream = torch.cuda.Stream(device=dev)
  main_stream = torch.cuda.current_stream()
  ready = [torch.cuda.Event() for _ in range(2)]   # stage[b] holds its batch
  freed = [torch.cuda.Event() for _ in range(2)]   # the encoder is done reading stage[b]

  def queue_h2d(i):
    b = i & 1
    with torch.cuda.stream(copy_stream):
      copy_stream.wait_event(freed[b])
      stages[b].copy_(ys_pinned[i % n_rot], non_blocking=True)
      ready[b].record(copy_stream)

  def e2e_run(k):
    nb = 0
    for b in range(2):
      freed[b].record(main_stream)
    queue_h2d(0)
    for i in range(k):
      b = i & 1
      if i + 1 < k:
        queue_h2d(i + 1)
      main_stream.wait_event(ready[b])
      s = model.compress(stages[b])
      freed[b].record(main_stream)
      nb = s.nbytes()
      host_bytes[b][:nb].copy_(s.bytes_dev[:nb], non_blocking=True)
      host_offs[b].copy_(s.offsets_dev, non_blocking=True)
    main_stream.synchronize()
    return nb

  e2e_run(3)
  e2e_ms = []
  for _ in range(E2E_REPEATS):
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    nb = e2e_run(args.steps)
    e1.record()
    barrier()
    e2e_ms.append(allmax(e0.elapsed_time(e1)))
  to_val = lambda ms: world * sym_per_step * args.steps / (ms * 1e-3) / 1e6
  e2e_value = to_val(float(np.median(e2e_ms)))

  result = {
      "metric": METRIC,
      "value": value, "unit": "Msymbols/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
      "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
      "dtype": "u32", "data": "synthetic",
      "config": {
          "workload": WORKLOAD,
          "bits_per_symbol": round(bits_per_symbol, 4), "streams_per_gpu": S, "symbols_per_stream": N,
          "l2": f"inputs rotate over {n_rot} distinct batches ({n_rot * 33.5:.0f} MB > 126 MB L2)",
          "parallelism": f"batch-shard x{world}, tables broadcast from rank 0",
          "tables_match_fixture": tables_match,
      },
      "value_repeats": {"median": float(np.median(vals)), "min": vals[0], "max": vals[-1], "regions": len(vals)},
      "e2e": {"value": e2e_value, "unit": "Msymbols/s", "h2d_bytes_per_step": int(world * ys[0].numel() * 4),
              "d2h_bytes_per_step": int(world * (nb + 8 * (S + 1))),
              "min": to_val(max(e2e_ms)), "max": to_val(min(e2e_ms)), "repeats": len(e2e_ms),
              "note": "median of the repeated K-step region; bytes summed over all ranks; H2D of batch i+1 overlaps "
                      "the encode of batch i (2 staging buffers)"},
      "gpu_launches": int(launches),
      "parity_checked": parity["all_ranks"], "parity": parity,
      "numa": numa,
  }

  if rank == 0:
    result["clocks"] = clocks.summary()

  phase("extras")
  if rank != 0:
    faulthandler.cancel_dump_traceback_later()   # waiting for rank 0's side measurements; torchrun ends us if it dies
  if rank == 0 and not args.no_extras:
    try:
      extras(result, model, ys, ys_host, strings, dev, args, sym_per_step, S, N)
    except Exception as e:  # pylint:disable=broad-except
      result["extras_error"] = repr(e)

  if rank == 0 and args.dump_outputs:
    dump_strings(args.dump_outputs, last_strings.tolist())
  if rank == 0:
    print(json.dumps(result))
  if world > 1:
    dist.barrier()
    dist.destroy_process_group()
  faulthandler.cancel_dump_traceback_later()


def extras(result, model, ys, ys_host, strings, dev, args, sym_per_step, S, N):
  """Side measurements of the same run (rank 0): dominant-kernel roofline, decode, cfg3, GDN, model path, CPU."""
  import torch
  import compression_b200 as tfc
  from compression_b200 import functional, gen_ops
  n_rot = CFG["n_rot"]
  peak, peak_src = _peaks()
  # --- dominant kernel of the step: the encode kernel, timed alone with events on the launch stream
  coff = model.cdf_offset.reshape(-1)
  qoff = model.quantization_offset
  lookup = model._lookup_host()
  times = []
  for i in range(8):
    h = gen_ops.create_range_encoder([S], lookup)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    functional.encode_channel_f32(h, ys[i % n_rot], qoff, coff)
    b.record()
    torch.cuda.synchronize()
    times.append(a.elapsed_time(b))
    h.close()
  enc_ms = float(np.median(times[2:]))
  alg_bytes = sym_per_step * 4 + strings.nbytes()
  achieved = alg_bytes / (enc_ms * 1e-3) / 1e9
  traffic, traffic_note = None, "no ncu capture of this build of the kernel"
  prof = os.path.join(ROOT, "profiles", "encode_kernel_traffic.json")
  if os.path.exists(prof):
    import hashlib
    with open(prof) as f:
      tj = json.load(f)
    src = os.path.join(ROOT, "compression_b200", "csrc", "range_coder.cu")
    cur = hashlib.sha256(open(src, "rb").read()).hexdigest()[:16] if os.path.exists(src) else None
    if tj.get("source_sha256_16") == cur:
      traffic, traffic_note = tj.get("dram_bytes_per_launch"), tj.get("note", "ncu --set full capture of this build")
    else:
      traffic_note = "profiles/encode_kernel_traffic.json was captured on another build of range_coder.cu: not reported"
  sm_clock = (result.get("clocks") or {}).get("sm_mhz") or 1965
  result["roofline"] = {
      "kernel": "encode_kernel (fused quantise + range encode; gather / chain / drain warps per stream)", "bound": "hbm",
      "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
      "traffic_note": traffic_note,
      "peak_source": peak_src, "kernel_ms": enc_ms, "algorithmic_bytes": alg_bytes,
      "kernel_msym_s": sym_per_step / (enc_ms * 1e-3) / 1e6,
      "chain_cycles_per_symbol": enc_ms * 1e-3 * sm_clock * 1e6 / N,
      "note": "latency-bound serial recurrence per stream (256 streams on 148 SMs); the HBM fraction is small by "
              "construction, chain_cycles_per_symbol is the figure that bounds it",
  }
  # --- decode path (create + fused decode/dequantise + finalize), same strings
  strings = model.compress(ys[0])
  dec_ms, out = _time_ms(lambda: model.decompress(strings, (CFG["hw"], CFG["hw"])), max(3, min(args.steps, 10)), warm=2)
  result["decode"] = {"value": sym_per_step / (dec_ms * 1e-3) / 1e6, "unit": "Msymbols/s", "ms_per_step": dec_ms,
                      "roundtrip_equals_quantize": bool(torch.equal(out, model.quantize(ys[0])))}
  if int(os.environ.get("WORLD_SIZE", "1")) > 1:
    # N > 1 is the scaling measurement: the other ranks wait at a barrier while rank 0 is here, so the long side
    # measurements (cfg3, GDN at 12 GiB tensors, the model path, the CPU baselines -- rank 0 at N = 1 only) stay
    # with the single-GPU run
    result["extras_note"] = "N > 1: cfg3 / GDN / model-path / CPU side measurements are taken by the N = 1 run"
    return
  # --- configs[2]: bmshj2018 hyperprior, both levels, encode and decode
  try:
    w = cfg3_workload(dev)
    em_y, em_z, y3, idx3, loc3, z3 = (w[k] for k in ("em_y", "em_z", "y", "idx", "loc", "z"))
    enc3 = lambda: (em_z.compress(z3), em_y.compress(y3, idx3, loc=loc3))
    sz, sy = enc3()
    dec3 = lambda: (em_z.decompress(sz, (4, 4)), em_y.decompress(sy, idx3, loc=loc3))
    res3 = {}
    nsym = y3.numel() + z3.numel()
    for name, fn in (("encode", enc3), ("decode", dec3)):
      ms, out3 = _time_ms(fn, 10)
      res3[name] = {"ms_per_step": ms, "value": nsym / (ms * 1e-3) / 1e6, "unit": "Msymbols/s"}
    zhat, yhat = out3
    res3["roundtrip_equals_quantize"] = bool(torch.equal(yhat, em_y.quantize(y3, loc3)) and torch.equal(zhat, em_z.quantize(z3)))
    res3["bits_per_symbol_y"] = 8.0 * sy.nbytes() / y3.numel()
    res3["workload"] = w["workload"]
    result["cfg3_bmshj2018"] = res3
    del w, y3, idx3, loc3, z3
  except Exception as e:  # pylint:disable=broad-except
    result["cfg3_bmshj2018"] = {"error": repr(e)}
  # --- GDN at the two analysis-transform shapes of cfg2 (forward) and backward at the first
  gdn = {}
  gamma = (0.1 * torch.eye(128) + (0.02 * torch.randn(128, 128)).abs()).to(dev)
  beta = (1 + 0.5 * torch.rand(128)).to(dev)
  for name, npix in (("gdn_0 [256,64,64,128]", 256 * 64 * 64), ("gdn_1 [256,32,32,128]", 256 * 32 * 32)):
    x = torch.randn(npix, 128, device=dev)
    ms, _ = _time_ms(lambda: functional.gdn_forward(x, gamma, beta), 10, warm=2)
    gbs = 8.0 * npix * 128 / (ms * 1e-3) / 1e9
    gdn[name] = {"fwd_ms": ms, "fwd_GBps": gbs, "fwd_frac_of_hbm_peak": gbs / peak}
    if npix == 256 * 64 * 64:
      dy = torch.randn_like(x)
      ms, _ = _time_ms(lambda: functional.gdn_backward(x, gamma, beta, dy), 7)
      gbs = 12.0 * npix * 128 / (ms * 1e-3) / 1e9
      gdn[name].update({"bwd_ms": ms, "bwd_GBps": gbs, "bwd_frac_of_hbm_peak": gbs / peak})
      del dy
    del x
  # --- configs[3]: GDN microbench, 192 channels, 64x64 tiles (batch 4096 if memory allows, else 1024)
  try:
    free_b, _ = torch.cuda.mem_get_info(dev)
    batch4 = 4096 if free_b > 90e9 else 1024
    npix = batch4 * 64 * 64
    gamma192 = (0.1 * torch.eye(192) + (0.02 * torch.randn(192, 192)).abs()).to(dev)
    beta192 = (1 + 0.5 * torch.rand(192)).to(dev)
    x = torch.randn(npix, 192, device=dev) * (0.05 + 3.95 * torch.rand(192, device=dev))  # SURVEY 8(d) cfg4 recipe
    ms, _ = _time_ms(lambda: functional.gdn_forward(x, gamma192, beta192), 5)
    gbs = 8.0 * npix * 192 / (ms * 1e-3) / 1e9
    entry = {"fwd_ms": ms, "fwd_GBps": gbs, "fwd_frac_of_hbm_peak": gbs / peak}
    torch.cuda.empty_cache()  # the forward's two cached 13 GB outputs
    dy = torch.randn_like(x)
    ms, _ = _time_ms(lambda: functional.gdn_backward(x, gamma192, beta192, dy), 3)
    gbs = 12.0 * npix * 192 / (ms * 1e-3) / 1e9
    entry.update({"bwd_ms": ms, "bwd_GBps": gbs, "bwd_frac_of_hbm_peak": gbs / peak})
    gdn[f"cfg4 [{batch4},64,64,192]"] = entry
    del x, dy
  except Exception as e:  # pylint:disable=broad-except
    gdn["cfg4 [4096,64,64,192]"] = {"error": repr(e)}
  result["gdn"] = gdn
  torch.cuda.empty_cache()
  # --- the model path as configs[1]/[2] name it: images -> analysis transform (conv glue + GDN) -> strings
  try:
    from compression_b200 import models
    result["model_path"] = models.bench_model_paths(dev)
  except Exception as e:  # pylint:disable=broad-except
    result["model_path"] = {"error": repr(e)}
  # --- CPU baselines on this box's host cores (bounded: one cfg2 batch; persistent worker pool)
  try:
    q = model.quantization_offset
    value_host = symbols_of(model.cdf_offset.cpu().numpy(), None if q is None else q.cpu(), ys_host[0])
    cores, phys = os.cpu_count() or 1, physical_cores()
    os.sched_setaffinity(0, range(cores)) if hasattr(os, "sched_setaffinity") else None  # un-pin: all host cores
    sweep, best_t = sweep_threads(value_host, lookup, cores)
    enc_best, dec_best, kind = cpu_coder_times(value_host, lookup, best_t)
    enc_all, dec_all, _ = cpu_coder_times(value_host, lookup, cores)
    enc_phys, dec_phys, _ = cpu_coder_times(value_host, lookup, phys)
    enc_one, dec_one, _ = cpu_coder_times(value_host[:16], lookup, 1, repeats=3)
    result["cpu_baseline"] = {
        "value": enc_best["median"], "unit": "Msymbols/s", "cores": best_t, "kind": kind,
        "sample": f"one full cfg2 batch ({S} streams x {N} int32 symbols), EntropyEncodeChannel+Finalize, median of 5 "
                  f"after warm-up, streams on a persistent pool of {best_t} threads (the fastest of the sweep "
                  f"1..{cores}; this box reports {cores} logical CPUs)",
        "thread_sweep_msym_s": {str(k): round(v, 1) for k, v in sweep.items()},
        "encode": {"threads_best": enc_best, "threads_all": enc_all, "threads_physical": enc_phys, "threads_1": enc_one},
        "decode": {"threads_best": dec_best, "threads_all": dec_all, "threads_physical": dec_phys, "threads_1": dec_one},
        "logical_cpus": cores, "physical_cores": phys, "single_core_value": enc_one["median"],
        "single_core_sample": "16 streams x 32768 symbols, 1 thread",
        "gdn_torch_cpu": cpu_gdn_baseline(),
    }
    result["speedup_vs_cpu"] = {
        "encode_vs_1_thread": result["value"] / enc_one["median"], "encode_vs_best_threads": result["value"] / enc_best["median"],
        "decode_vs_1_thread": result["decode"]["value"] / dec_one["median"],
        "decode_vs_best_threads": result["decode"]["value"] / dec_best["median"],
    }
  except Exception as e:  # pylint:disable=broad-except
    result["cpu_baseline"] = {"error": repr(e)}


if __name__ == "__main__":
  main()
