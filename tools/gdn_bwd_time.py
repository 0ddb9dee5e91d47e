"""Tensor-core GDN backward across builds of the library: time per call, kernels launched, and outputs.

  python tools/gdn_bwd_time.py --libs OLD.so NEW.so --out DIR [--rounds 2] [--b192 4096]

For each round, each library runs in turn in a fresh process (TFCB_LIB_PATH), so that two builds are compared
alternately on the same GPU.  A process times F.gdn_backward at [256,64,64,128] and [B,64,64,192] for the default GDN
(alpha = 1, epsilon = 1, no rectification: FAST) and for every other flag combination the tensor cores take
(alpha in {1, 2} x epsilon in {1, 1/2} x rectify), each as GDN and IGDN: the median of per-call CUDA event times
after warm-up.  In the first two rounds each process then runs an untimed pass that lists the kernels every case
launches (torch.profiler) and writes the outputs of seeded inputs at [256,64,64,C] to DIR: dgamma and dbeta whole,
dx as a strided sample and, for FAST, a SHA-256 digest.  The second round gives each build's own run-to-run
difference.  The summary compares every library's outputs with those of the first library's first round.
"""
import argparse, hashlib, json, os, subprocess, sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = [(a, e, r) for a in (1.0, 2.0) for e in (1.0, 0.5) for r in (False, True)]  # (1, 1, False) is FAST


def _inputs(torch, C, n_pix):
  g = torch.Generator(device="cuda").manual_seed(C)
  gamma = 0.1 * torch.eye(C, device="cuda") + (0.02 * torch.randn(C, C, device="cuda", generator=g)).abs()
  beta = 1 + 0.5 * torch.rand(C, device="cuda", generator=g)
  x = torch.randn(n_pix, C, device="cuda", generator=g) * (0.05 + 3.95 * torch.rand(C, device="cuda", generator=g))
  x[::7, ::5] = 0.0  # exact zeros: the pool's derivative is 0 there
  dy = torch.randn(n_pix, C, device="cuda", generator=g)
  return x, gamma, beta, dy


def _key(C, alpha, eps, rect, inv):
  return f"C={C} alpha={alpha:g} eps={eps:g} rectify={int(rect)} inverse={int(inv)}"


def worker(args):
  import torch
  sys.path.insert(0, ROOT)
  from compression_b200 import functional as F
  out = {"lib": os.environ["TFCB_LIB_PATH"], "gpu": torch.cuda.get_device_name(0), "ms": {}}
  smi = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
  out["power_limit_and_max_sm_clock"] = smi.stdout.strip().splitlines()[0] if smi.returncode == 0 else "unknown"
  for C, B in ((128, 256), (192, args.b192)):
    x, gamma, beta, dy = _inputs(torch, C, B * 64 * 64)
    for alpha, eps, rect in CASES:
      for inv in (False, True):
        fn = lambda: F.gdn_backward(x, gamma, beta, dy, inv, rect, alpha, eps)
        for _ in range(3):
          fn()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.reps)]
        torch.cuda.synchronize()
        for i in range(args.reps):
          ev[2 * i].record()
          fn()
          ev[2 * i + 1].record()
        torch.cuda.synchronize()
        ts = sorted(ev[2 * i].elapsed_time(ev[2 * i + 1]) for i in range(args.reps))
        out["ms"][_key(C, alpha, eps, rect, inv)] = ts[args.reps // 2]
    del x, dy
    torch.cuda.empty_cache()
  if args.dump:
    from torch.profiler import profile, ProfilerActivity
    out["kernels"], arrays = {}, {}
    for C in (128, 192):
      x, gamma, beta, dy = _inputs(torch, C, 256 * 64 * 64)
      for alpha, eps, rect in CASES:
        for inv in (False, True):
          key = _key(C, alpha, eps, rect, inv)
          torch.cuda.synchronize()
          with profile(activities=[ProfilerActivity.CUDA]) as prof:
            dx, dg, db = F.gdn_backward(x, gamma, beta, dy, inv, rect, alpha, eps)
            torch.cuda.synchronize()
          names = {e.name.split("(")[0] for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
          out["kernels"][key] = sorted(names)
          if (alpha, eps, rect) == CASES[0]:
            arrays[key + " dx_sha256"] = hashlib.sha256(dx.cpu().numpy().tobytes()).hexdigest()
          arrays[key + " dx_sample"] = dx.reshape(-1)[::9973].cpu().numpy()
          arrays[key + " dgamma"] = dg.cpu().numpy()
          arrays[key + " dbeta"] = db.cpu().numpy()
      del x, dy
      torch.cuda.empty_cache()
    import numpy as np
    np.savez(args.dump, **{k: np.asarray(v) for k, v in arrays.items()})
  print(json.dumps(out), flush=True)


def _compare(ref, other):
  """Per case of two dumps: (case, dx bit-identical or None where no digest was kept, max |difference| of the dx
  sample, of dgamma, of dbeta)."""
  import numpy as np
  a, b = np.load(ref), np.load(other)
  rows = []
  for k in sorted(x[: -len(" dgamma")] for x in a.files if x.endswith(" dgamma")):
    same = str(a[k + " dx_sha256"]) == str(b[k + " dx_sha256"]) if k + " dx_sha256" in a.files else None
    diff = [float(np.abs(a[k + t].astype(np.float64) - b[k + t]).max()) for t in (" dx_sample", " dgamma", " dbeta")]
    rows.append((k, same, *diff))
  return rows


def main():
  ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
  ap.add_argument("--libs", nargs="+", help="library paths, compared in this order")
  ap.add_argument("--rounds", type=int, default=2)
  ap.add_argument("--reps", type=int, default=7, help="timed calls per case")
  ap.add_argument("--b192", type=int, default=4096, help="batch of the timed C = 192 shape [B,64,64,192]")
  ap.add_argument("--out", help="directory for the outputs and runs.json")
  ap.add_argument("--dump", help=argparse.SUPPRESS)  # worker: .npz path for the outputs
  ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
  args = ap.parse_args()
  if args.worker:
    return worker(args)
  if not args.libs or not args.out:
    ap.error("--libs and --out are required")
  os.makedirs(args.out, exist_ok=True)
  runs = []  # (lib index, round, result)
  for rnd in range(args.rounds):
    for i, lib in enumerate(args.libs):
      cmd = [sys.executable, os.path.abspath(__file__), "--worker", "--reps", str(args.reps), "--b192", str(args.b192)]
      if rnd < 2:  # two dumps per library: the second gives the build's own run-to-run difference
        cmd += ["--dump", os.path.join(args.out, f"lib{i}_r{rnd}.npz")]
      p = subprocess.run(cmd, env=dict(os.environ, TFCB_LIB_PATH=os.path.abspath(lib)), capture_output=True, text=True)
      if p.returncode != 0:
        sys.exit(f"{lib} round {rnd} failed:\n{p.stderr[-4000:]}")
      res = json.loads(p.stdout.strip().splitlines()[-1])
      runs.append((i, rnd, res))
      print(f"[lib{i} round {rnd}] {lib}: {res['gpu']}, power limit / max SM clock {res['power_limit_and_max_sm_clock']}",
            flush=True)
      if "kernels" in res and rnd == 0:
        for k, names in res["kernels"].items():
          print(f"  kernels  {k}: {', '.join(names)}")
  with open(os.path.join(args.out, "runs.json"), "w") as f:
    json.dump([{"lib": args.libs[i], "round": r, **res} for i, r, res in runs], f, indent=1)
  keys = list(runs[0][2]["ms"])
  print("\nmedian ms per call (every round)")
  for k in keys:
    cols = "  |  ".join(f"lib{i}: " + " ".join(f"{res['ms'][k]:7.3f}" for j, _, res in runs if j == i)
                        for i in range(len(args.libs)))
    print(f"  {k:45s} {cols}")
  ref = os.path.join(args.out, "lib0_r0.npz")
  for i in range(len(args.libs)):
    for rnd in range(2):
      other = os.path.join(args.out, f"lib{i}_r{rnd}.npz")
      if (i, rnd) == (0, 0) or not os.path.exists(other):
        continue
      print(f"\noutputs of lib{i} round {rnd} against lib0 round 0")
      for k, same, dxs, dg, db in _compare(ref, other):
        tag = "" if same is None else ("dx bit-identical" if same else "dx DIFFERS")
        print(f"  {k:45s} {tag:17s} max|d| dx sample {dxs:.2e}  dgamma {dg:.2e}  dbeta {db:.2e}")

if __name__ == "__main__":
  main()
