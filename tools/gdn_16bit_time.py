"""16-bit GDN activations: the native kernels against the conversion path, in one process.

  python tools/gdn_16bit_time.py --out FILE.json [--reps 9] [--b192 4096] [--dtype bfloat16]

The conversion path is what a 16-bit call did before the kernels read 16-bit elements themselves: widen x (and dy) to
float32, run the float32 kernels, round y (dx) back.  Cases: forward at [B,64,64,192], backward at [256,64,64,128]
and at [B,64,64,192] (B = 4096 is cfg4's batch; if the card has too little free memory for both arms the script
retries with B = 1024 and says so in the output).  Per case: the median of per-call CUDA event times after warm-up,
the two arms alternating call by call; the peak of torch.cuda.max_memory_allocated() above the inputs during one call
of each arm; the rate on the algorithmic scale (forward: x in, y out, 4 B/element; backward: x, dy in, dx out,
6 B/element); and whether the two arms agree (y, dx bit-identical; dgamma, dbeta within 1e-6 of their largest entry).
The card's name, power limit and maximum SM clock go into the JSON beside the numbers.
"""
import argparse, json, os, subprocess, sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _inputs(torch, C, n_pix, dtype):
  g = torch.Generator(device="cuda").manual_seed(C)
  gamma = 0.1 * torch.eye(C, device="cuda") + (0.02 * torch.randn(C, C, device="cuda", generator=g)).abs()
  beta = 1 + 0.5 * torch.rand(C, device="cuda", generator=g)
  x = (torch.randn(n_pix, C, device="cuda", generator=g) *
       (0.05 + 3.95 * torch.rand(C, device="cuda", generator=g))).to(dtype)
  x[::7, ::5] = 0.0
  dy = torch.randn(n_pix, C, device="cuda", generator=g).to(dtype)
  return x, gamma, beta, dy


def _of_max(a, b):
  return float((a.double() - b.double()).abs().max() / b.double().abs().max())


def run_case(torch, F, direction, C, batch, dtype, reps):
  n_pix = batch * 64 * 64
  x, gamma, beta, dy = _inputs(torch, C, n_pix, dtype)
  if direction == "forward":
    native = lambda: F.gdn_forward(x, gamma, beta)
    convert = lambda: F.gdn_forward(x.float(), gamma, beta).to(dtype)
    bytes_per_elem = 4
  else:
    native = lambda: F.gdn_backward(x, gamma, beta, dy)

    def convert():
      dx, dg, db = F.gdn_backward(x.float(), gamma, beta, dy.to(torch.float32))
      return dx.to(dtype), dg, db
    bytes_per_elem = 6
  res = {"direction": direction, "shape": [batch, 64, 64, C], "dtype": str(dtype).replace("torch.", "")}
  # outputs of the two arms, then the peak memory of one call of each
  a, b = native(), convert()
  if direction == "forward":
    res["outputs_agree"] = bool(torch.equal(a, b))
  else:
    res["dx_bit_identical"] = bool(torch.equal(a[0], b[0]))
    res["dgamma_of_max"], res["dbeta_of_max"] = _of_max(a[1], b[1]), _of_max(a[2], b[2])
    res["outputs_agree"] = res["dx_bit_identical"] and res["dgamma_of_max"] <= 1e-6 and res["dbeta_of_max"] <= 1e-6
  del a, b
  for name, fn in (("native", native), ("conversion", convert)):
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out = fn()
    torch.cuda.synchronize()
    res[f"{name}_peak_gb"] = (torch.cuda.max_memory_allocated() - base) / 1e9
    del out
  # timing: warm-up, then the arms alternate call by call
  for _ in range(2):
    native(), convert()
  ts = {"native": [], "conversion": []}
  for _ in range(reps):
    for name, fn in (("native", native), ("conversion", convert)):
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      torch.cuda.synchronize()
      e0.record()
      out = fn()
      e1.record()
      torch.cuda.synchronize()
      ts[name].append(e0.elapsed_time(e1))
      del out
  algo_bytes = bytes_per_elem * n_pix * C
  for name, t in ts.items():
    med = sorted(t)[len(t) // 2]
    res[f"{name}_ms"] = med
    res[f"{name}_ms_all"] = t
    res[f"{name}_gbps_algorithmic"] = algo_bytes / (med * 1e-3) / 1e9
  res["speedup"] = res["conversion_ms"] / res["native_ms"]
  del x, dy
  torch.cuda.empty_cache()
  return res


def main():
  ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
  ap.add_argument("--out", required=True, help="JSON file for the results")
  ap.add_argument("--reps", type=int, default=9, help="timed calls per arm and case")
  ap.add_argument("--b192", type=int, default=4096, help="batch of the C = 192 shape [B,64,64,192]")
  ap.add_argument("--dtype", choices=["bfloat16", "float16"], default="bfloat16")
  args = ap.parse_args()
  import torch
  sys.path.insert(0, ROOT)
  from compression_b200 import functional as F
  if not torch.cuda.is_available():
    sys.exit("gdn_16bit_time.py measures on a CUDA device; none is available")
  dtype = getattr(torch, args.dtype)
  smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
  out = {"gpu": torch.cuda.get_device_name(0),
         "nvidia_smi_name_power_limit_max_sm_clock": smi.stdout.strip().splitlines()[0] if smi.returncode == 0 else "unknown",
         "cases": [], "notes": []}
  for direction, C, batch in (("backward", 128, 256), ("forward", 192, args.b192), ("backward", 192, args.b192)):
    res = None
    try:
      res = run_case(torch, F, direction, C, batch, dtype, args.reps)
    except torch.cuda.OutOfMemoryError:
      pass
    if res is None:  # (retried outside the handler, whose traceback still holds the first attempt's tensors)
      torch.cuda.empty_cache()
      out["notes"].append(f"{direction} C={C}: out of memory at batch {batch}, measured at batch 1024 instead")
      res = run_case(torch, F, direction, C, 1024, dtype, args.reps)
    out["cases"].append(res)
    print(f"{direction:8s} {res['shape']} {res['dtype']}: native {res['native_ms']:.3f} ms "
          f"({res['native_gbps_algorithmic']:.0f} GB/s, peak {res['native_peak_gb']:.2f} GB)  conversion "
          f"{res['conversion_ms']:.3f} ms ({res['conversion_gbps_algorithmic']:.0f} GB/s, peak {res['conversion_peak_gb']:.2f} GB)"
          f"  x{res['speedup']:.2f}  outputs agree: {res['outputs_agree']}", flush=True)
  print(out["gpu"], "|", out["nvidia_smi_name_power_limit_max_sm_clock"], *out["notes"], sep="\n")
  os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
  with open(args.out, "w") as f:
    json.dump(out, f, indent=1)


if __name__ == "__main__":
  main()
