"""Device time of the per-column droplet-number step (kidmp_step_device_nc) against the plain step (kidmp_step_device).

Two workloads, device events on one torch stream, median over --repeats rounds after --warmup:

  bench   the bench domain (--columns x 60 levels, dt = 10 s) stepped --steps times in a row from the same start, by one handle
          with the plain step and with per-column values (eight values in a seeded shuffle); the two run alternately, round
          by round.  Reported per step.
  sweep   a KiD-sized set_Nc sweep: eight values x 120 columns x 120 levels, as ONE per-column call over 960 columns of one
          handle, against eight handles (one per value) stepping their 120 columns one after the other.  Reported per sweep
          (all eight values once).

Every round restores the inputs outside the timed region.  Prints the GPU's name and power limit, then one JSON line.

    python tools/column_nc_time.py [--columns 1048576] [--steps 10] [--repeats 5] [--warmup 2] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

VALUES = np.array([10.0, 50.0, 100.0, 300.0, 400.0, 1000.0, 2000.0, 3000.0], np.float32)


def gpu_identity():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                       # (the figure is then reported as unknown, never guessed)
        pl = "unknown (%s)" % e
    return name, pl


class Domain:
    """Device inputs of one workload ([nz][ncol] tensors; c0:c1 takes those columns as arrays of their own) and their working
    copies."""

    def __init__(self, src, p, dz, c0=0, c1=None):
        import torch
        cut = lambda a: a[:, c0:c1].contiguous()
        self.src, self.p, self.dz = {k: cut(v) for k, v in src.items()}, cut(p), dz
        self.st = {k: v.clone() for k, v in self.src.items()}
        self.nz, self.ncol = self.p.shape
        self.ppt = torch.zeros((4, self.ncol), dtype=torch.float32, device="cuda")

    def reset(self):
        for k, v in self.src.items():
            self.st[k].copy_(v)

    def step(self, th, dt, stream, set_nc=None):
        from kid_b200.kidmp import FIELDS
        th.step_device(self.ncol, self.nz, dt, [self.st[k].data_ptr() for k in FIELDS], self.p.data_ptr(), self.dz.data_ptr(),
                       self.ppt.data_ptr(), stream=stream, set_nc_ptr=set_nc)


def timed(stream, fn):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    fn()
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--columns", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    from kid_b200 import synth
    from kid_b200.kidmp import Thompson
    if not torch.cuda.is_available():
        raise SystemExit("column_nc_time.py: no CUDA device")
    name, power = gpu_identity()
    print("GPU: %s, power limit %s" % (name, power))
    s = torch.cuda.Stream()
    sp = s.cuda_stream
    res = {"gpu": name, "power_limit": power}

    # bench domain: plain and per-column steps of one handle, alternately
    th = Thompson(set_Nc=100.0, iiwarm=False, l_sediment=True)
    d = Domain(*synth.make_domain(args.columns, nz=60, nx=1024, device="cuda"))
    nc = torch.from_numpy(VALUES[np.random.default_rng(1).permutation(np.arange(d.ncol) % 8)]).cuda()
    runs = {"plain": None, "per_column": nc.data_ptr()}
    ms = {k: [] for k in runs}
    torch.cuda.synchronize()
    for r in range(args.warmup + args.repeats):
        for k, ptr in runs.items():
            d.reset()
            torch.cuda.synchronize()
            t = timed(s, lambda: [d.step(th, 10.0, sp, set_nc=ptr) for _ in range(args.steps)])
            if r >= args.warmup:
                ms[k].append(t / args.steps)
    res["bench"] = {"columns": d.ncol, "levels": 60, "steps": args.steps,
                    **{k + "_ms_per_step": float(np.median(v)) for k, v in ms.items()},
                    **{k + "_ms_all": [round(x, 4) for x in v] for k, v in ms.items()}}
    b = res["bench"]
    print("bench %d x 60: plain %.3f ms/step, per-column %.3f ms/step (%+.2f %%)" % (
        d.ncol, b["plain_ms_per_step"], b["per_column_ms_per_step"], 100.0 * (b["per_column_ms_per_step"] / b["plain_ms_per_step"] - 1.0)))
    del d, nc
    th.close()

    # KiD-sized sweep: 8 values x 120 columns x 120 levels
    per = 120
    src = synth.make_domain(len(VALUES) * per, nz=120, nx=1024, device="cuda", cloudy_fraction=1.0)
    d = Domain(*src)
    parts = [Domain(*src, c0=i * per, c1=(i + 1) * per) for i in range(len(VALUES))]       # the same columns, value by value
    one = Thompson(set_Nc=100.0, iiwarm=False, l_sediment=True)
    eight = [Thompson(set_Nc=float(v), iiwarm=False, l_sediment=True) for v in VALUES]
    nc = torch.from_numpy(np.repeat(VALUES, per)).cuda()
    ways = {"one_call": lambda: d.step(one, 10.0, sp, set_nc=nc.data_ptr()),
            "eight_handles": lambda: [q.step(h, 10.0, sp) for q, h in zip(parts, eight)]}
    ms = {k: [] for k in ways}
    torch.cuda.synchronize()
    for r in range(args.warmup + 20 * args.repeats):
        for k, fn in ways.items():
            for q in [d] + parts:
                q.reset()
            torch.cuda.synchronize()
            t = timed(s, fn)
            if r >= args.warmup:
                ms[k].append(t)
    res["sweep"] = {"values": len(VALUES), "columns_per_value": per, "levels": 120,
                    **{k + "_ms": float(np.median(v)) for k, v in ms.items()}}
    w = res["sweep"]
    print("sweep 8 x %d x 120: one per-column call %.3f ms, eight handles %.3f ms" % (per, w["one_call_ms"], w["eight_handles_ms"]))
    for h in eight + [one]:
        h.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
