#!/usr/bin/env python
"""bench.py - column-steps/s of the Thompson microphysics step on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun)
    python bench.py --impl reference ...                     (the reference's CPU path: the oracle)
    python bench.py ... --dump-outputs DIR                   (also write the outputs of the last timed step, to compare two builds)

Workload (BASELINE.json configs[3]): synthetic 1024x1024 = 1 048 576 columns x 60 levels per GPU from
the seeded CONUS-like convective domain of kid_b200/synth.py (about 30 % cloudy columns), dt = 10 s.
Default = weak scaling: every rank owns its own 1 048 576 columns [rank*ncol, (rank+1)*ncol) of one global
domain.  --total-columns N = strong scaling (BASELINE.json configs[4]: N = 16 777 216 = 4096x4096): the N columns of one
domain are cut into contiguous shards, one per rank (kid_b200/shard.py).  Columns are independent, so there is no
data-path collective - NCCL only reduces the eight domain diagnostics once per run.

A "step" = one kidmp_step_device call over all resident columns: classification, work list and sorted list of the busy
cells, the four cell kernels (S1..S13 of every busy cell), what runs down the columns, sedimentation + final clamps,
ordered domain sums (15 launches per chunk of 1 048 576 columns); the state evolves in place from step to step like a
model time loop.  Inputs (2.8 GB per GPU) are far larger than L2, so no flush is needed between steps.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "column-steps/sec (60-lev Thompson)"
UNIT = "column-steps/s"
ALG_BYTES_PER_COLUMN = 4576          # SURVEY.md section 8(d): 10 fields read + 9 written + 4 precip scalars, nz=60
NZ = 60
DT = 10.0
# dram__bytes_read.sum + dram__bytes_write.sum of the kernels of one step of this workload, from the committed ncu launch
# list of this round (profiles/r02_traffic.json, written by tools/ncu_traffic.py from the CSV next to it)
TRAFFIC_FILE = os.path.join(ROOT, "profiles", "r02_traffic.json")


def measured_traffic():
    try:
        with open(TRAFFIC_FILE) as f:
            t = json.load(f)
        return float(t["bytes_per_step"]), {"file": "profiles/r02_traffic.json", "commit": t.get("commit"), "per_kernel_MB": t.get("per_kernel_MB")}
    except Exception as e:
        return None, {"file": "profiles/r02_traffic.json", "error": str(e)}


def fortran_probe():
    """Is there a Fortran compiler on this box (BASELINE.md section 3.2)?  With one, oracle/ref builds the reference itself."""
    import shutil
    tried = ("gfortran", "flang", "flang-new", "nvfortran", "ifx", "ifort", "f95", "pgfortran")
    found = [c for c in tried if shutil.which(c)]
    return {"found": found, "tried": list(tried)}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the GPU is under load (B200_PROFILING.md recipe): one
    streaming `nvidia-smi -lms 100` process, started before the warm-up so that samples exist inside a
    timed region of a few hundred milliseconds; `mark()` brackets the timed region."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.t0 = self.t1 = None
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                parts = [x.strip() for x in line.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append((time.perf_counter(), parts))
        except Exception:
            pass

    def mark(self, start):
        if start:
            self.t0 = time.perf_counter()
        else:
            self.t1 = time.perf_counter()

    def summary(self):
        if self.proc is not None:
            try:
                self.proc.terminate()
                self.proc.wait(timeout=10)         # reaped here: no defunct nvidia-smi outlives the run
            except Exception:
                pass
        inside = [r for t, r in self.rows if self.t0 is not None and self.t0 <= t <= (self.t1 or 1e99)]
        where = "timed region"
        if not inside:                 # region shorter than the sampling period: samples of the warm-up just before it
            inside = [r for t, r in self.rows if self.t0 is None or t <= self.t0][-5:]
            where = "warm-up just before the timed region"
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in inside)
        reasons = []
        for j, name in ((3, "hw_slowdown"), (4, "hw_thermal_slowdown"), (5, "sw_thermal_slowdown"), (6, "sw_power_cap")):
            if any(r[j].lower().startswith("active") for r in inside):
                reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(inside[0][1]), "reasons": reasons,
                "samples": len(inside), "sampled_in": where, "power_w_max": max(float(r[2]) for r in inside)}


def cpu_reference_run(ncol, steps, warmup, nthreads, col0=0):
    """The reference's CPU path (the C++ restatement under oracle/: no Fortran compiler exists here)
    on `ncol` columns of the bench domain, all host threads.  Returns (column-steps/s, ms/step, init_s)."""
    from kid_b200 import synth
    # the oracle keeps its collection tables between runs; the tree may be read-only, so they go to a per-user temporary directory
    os.environ.setdefault("KOR_CACHE_DIR", os.path.join(tempfile.gettempdir(), "kid_b200_oracle_cache_%d" % os.getuid()))
    from oracle.oracle import Oracle
    o = Oracle(set_Nc=100.0, iiwarm=False, l_sediment=True, nthreads=nthreads)
    st, p, dz = synth.make_domain(ncol, nz=NZ, col0=col0, nx=1024)
    state = {k: v.numpy().copy() for k, v in st.items()}
    pn, dzn = p.numpy().copy(), dz.numpy().copy()
    for _ in range(warmup):
        o.step(DT, state, pn, dzn, nthreads=nthreads)
    t0 = time.perf_counter()
    for _ in range(steps):
        o.step(DT, state, pn, dzn, nthreads=nthreads)
    el = time.perf_counter() - t0
    init_s = o.init_seconds
    o.close()
    return ncol * steps / el, el / steps * 1e3, init_s


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    ncol = args.cpu_columns
    probe = fortran_probe()
    v, ms, init_s = cpu_reference_run(ncol, args.steps, args.warmup, cores)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32+f64", "data": "synthetic",
        "config": {"workload": "synthetic 1024x1024 columns x 60 levels, CONUS-like convective domain, dt=10s",
                   "sample_columns": ncol, "nz": NZ, "dt": DT},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "fortran_probe": probe,
                         "sample": "first %d columns of the bench domain x %d steps (a rate: the full workload has 1 048 576), "
                                   "OpenMP over columns on %d threads; C++ restatement of the reference built -O3 without "
                                   "fast-math (no Fortran compiler on this box: see fortran_probe), table init %.1f s excluded"
                                   % (ncol, args.steps, cores, init_s)},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


DUMP_COLUMNS = 24576                 # --dump-outputs: 2176 bytes a column (nine fields of 60 levels + 4 precipitation amounts) = 53.5 MB
DUMP_SEED = 20261018


def dump_outputs(out_dir, st, ppt, ncol):
    """What the last timed step returned to the caller: the nine state fields (NZ, ncol) and the surface precipitation of the step
    (4, ncol), as <out_dir>/<name>.npy in float32.  A domain of more than DUMP_COLUMNS columns is cut to a seeded sample of
    columns (sorted, the same in every run), so that two builds of the project can be compared output for output."""
    import torch
    from kid_b200.kidmp import FIELDS
    cols = np.arange(ncol) if ncol <= DUMP_COLUMNS else np.sort(np.random.default_rng(DUMP_SEED).choice(ncol, DUMP_COLUMNS, replace=False))
    idx = torch.from_numpy(cols).to(ppt.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in [(k, st[k]) for k in FIELDS] + [("ppt", ppt)]:
        np.save(os.path.join(out_dir, name + ".npy"), a.index_select(1, idx).cpu().numpy())


def make_resident_domain(synth, ncol, col0, nx, dev, slab=1 << 20):
    """kid_b200/synth.py domain [col0, col0+ncol) on the device, generated slab by slab into preallocated tensors."""
    import torch
    from kid_b200.kidmp import FIELDS
    st = {k: torch.empty((NZ, ncol), dtype=torch.float32, device=dev) for k in FIELDS}
    p = torch.empty((NZ, ncol), dtype=torch.float32, device=dev)
    dz = None
    for c in range(0, ncol, slab):
        n = min(slab, ncol - c)
        s1, p1, dz = synth.make_domain(n, nz=NZ, col0=col0 + c, nx=nx, device=dev)
        for k in FIELDS:
            st[k][:, c:c + n] = s1[k]
        p[:, c:c + n] = p1
        del s1, p1
    return st, p, dz


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="kidmp", choices=["kidmp", "reference"])
    ap.add_argument("--columns", type=int, default=1024 * 1024, help="columns per GPU (weak scaling)")
    ap.add_argument("--total-columns", type=int, default=0, help="columns of the whole domain, sharded over the GPUs (strong scaling)")
    ap.add_argument("--cpu-columns", type=int, default=262144, help="columns of the bounded CPU sample")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned on rank 0 (state fields and "
                    "surface precipitation, a fixed sample of %d columns) as DIR/<name>.npy" % DUMP_COLUMNS)
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "kidmp" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from kid_b200 import synth
    from kid_b200.kidmp import Thompson, FIELDS

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the kidmp arm has no CPU path (use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from kid_b200.shard import bind_to_gpu_numa
    numa = bind_to_gpu_numa(local)                       # before any pinned allocation: the staging arrays go to the GPU's node
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    strong = args.total_columns > 0
    if strong:
        from kid_b200.shard import shard_range
        col0, col1 = shard_range(args.total_columns, rank, world)
        ncol, nxdom = col1 - col0, int(round(args.total_columns ** 0.5))
    else:
        ncol, col0, nxdom = args.columns, rank * args.columns, 1024
    total_cols = args.total_columns if strong else world * ncol
    th = Thompson(set_Nc=100.0, iiwarm=False, l_sediment=True, device=local)
    # synthetic state generated directly in HBM, this rank's shard of the global domain (in slabs: the generator's temporaries)
    st, p, dz = make_resident_domain(synth, ncol, col0, nxdom, dev)
    presence = synth.stats(st)
    ppt = torch.zeros((4, ncol), dtype=torch.float32, device=dev)
    tstream = torch.cuda.Stream(device=dev)             # the launching stream: kernels and timing events both go here
    torch.cuda.synchronize()
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0
    fptr = [st[k].data_ptr() for k in FIELDS]

    def one_step():
        th.step_device(ncol, NZ, DT, fptr, p.data_ptr(), dz.data_ptr(), ppt.data_ptr(), stream=stream)

    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(args.warmup):
        one_step()
    torch.cuda.synchronize()
    th.diag()
    launches0 = th.gpu_launches

    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.mark(True)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    for i in range(args.steps):
        ev[i].record()
        one_step()
    ev[args.steps].record()
    torch.cuda.synchronize()
    sampler.mark(False)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, st, ppt, ncol)
    diag = torch.from_numpy(th.diag()).to(dev)          # the 8 domain sums accumulated over the K steps
    if world > 1:
        dist.all_reduce(diag)                           # the only collective: 64 bytes of diagnostics
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    total_ms = ev[0].elapsed_time(ev[args.steps])
    per_step = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    clocks = sampler.summary()
    launches = th.gpu_launches - launches0

    tmax = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    total_ms = float(tmax.item())
    ms_per_step = total_ms / args.steps
    value = total_cols * args.steps / (total_ms * 1e-3)
    stats = th.step_stats()
    # per-kernel device times: three more steps with the kernels of a launch one after the other and an event after each
    th.set_option("timing", 1)
    kms = {}
    for _ in range(3):
        one_step()
        torch.cuda.synchronize()
        for k, v in th.last_kernel_ms().items():
            kms[k] = kms.get(k, 0.0) + v / 3.0
    th.set_option("timing", 0)

    # ---- end to end through the C ABI with pinned HOST buffers (H2D + kernel + D2H every step) --------
    e2e = None
    if args.e2e_steps > 0:
        ncol_full = ncol
        ncol = min(ncol, 1 << 20)                        # strong scaling with larger shards: the first 1 048 576 columns of the shard
        host = {k: torch.empty((NZ, ncol), dtype=torch.float32).pin_memory() for k in FIELDS}
        del st, p
        st0, p0, dz0 = make_resident_domain(synth, ncol, col0, nxdom, dev)
        for k in FIELDS:
            host[k].copy_(st0[k])
        hp = torch.empty((NZ, ncol), dtype=torch.float32).pin_memory()
        hp.copy_(p0)
        del st0, p0
        hstate = {k: host[k].numpy() for k in FIELDS}
        hpn, hdz = hp.numpy(), dz0.cpu().numpy()
        th.step(DT, hstate, hpn, hdz)                    # warm-up (allocates the resident buffers)
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            th.step(DT, hstate, hpn, hdz)
        el = time.perf_counter() - t0
        tm = torch.tensor([el], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        el = float(tm.item())
        zc = bool(th.step_stats().get("zero_copy_return"))
        dsum = th.diag()                                 # sums over the e2e steps (warm-up included): changed columns per step
        changed = int(round(dsum[6] / max(dsum[7], 1.0) * ncol))
        e2e = {"value": world * ncol * args.e2e_steps / el, "unit": UNIT,
               "h2d_bytes_per_step": int(ncol * NZ * 4 * 10 + NZ * 4),
               "d2h_bytes_per_step": int((changed if zc else ncol) * NZ * 4 * 9 + ncol * 16),
               "steps": args.e2e_steps, "ms_per_step": el / args.e2e_steps * 1e3, "columns_per_gpu": ncol,
               "api": "kidmp_step (host arrays, COL_FASTEST, pinned)", "numa": numa,
               "d2h": ("only the %d columns the step changed come back (clear-sky columns return bit for bit as they went in, M:1540), "
                       "written by a kernel into the pinned host arrays" % changed) if zc else "all columns copied back"}
        ncol = ncol_full

    if rank == 0:
        peak, peak_src = peaks()
        kern_ms = float(np.mean(per_step))
        achieved = ALG_BYTES_PER_COLUMN * ncol / (kern_ms * 1e-3) / 1e9
        traffic, traffic_src = measured_traffic()
        if ncol != 1048576:
            traffic, traffic_src = None, {"note": "measured for the 1 048 576-column workload only"}
        # algorithmic bytes of the streaming kernels (the cell kernels are bound by instruction issue, not by memory):
        # classification reads the ten fields of every column; the finish kernels read them again and write nine for the
        # cloudy columns; per busy cell a 128-byte record is written once and read 1.5 times
        busy, cloudy = stats["busy_cells"], stats["cloudy_columns"]
        ksum = sum(kms.values()) or 1.0
        kalg = {"classify": 40.0 * NZ * ncol, "carries": 64.0 * busy, "finish": (76.0 * NZ + 16.0) * cloudy + 128.0 * busy}
        kernels = {k: {"ms": round(v, 4), "share": round(v / ksum, 4)} for k, v in kms.items()}
        for k, b in kalg.items():
            if kms.get(k):
                kernels[k]["alg_bytes"] = b
                kernels[k]["frac"] = round(b / (kms[k] * 1e-3) / 1e9 / peak, 4)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "f32+f64", "data": "synthetic",
            "config": {"workload": ("synthetic %d columns x 60 levels sharded over the GPUs" % total_cols if strong else
                                    "synthetic 1024x1024 columns x 60 levels per GPU") + ", CONUS-like convective domain "
                                   "(kid_b200/synth.py seed 20261018), dt=10s, state evolves in place",
                       "columns_per_gpu": ncol, "total_columns": total_cols, "nz": NZ, "dt": DT,
                       "l2": "inputs (2.8 GB per 1 048 576 columns) larger than L2, no flush",
                       "presence": presence, "step_stats_rank0_last_chunk": stats,
                       "active_column_fraction": float(diag[6].item() / max(diag[7].item(), 1.0))},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "kernel": "one step = the fifteen launches of kidmp_step_device (cell kernels k_cells<warm|ice|mixed|full> "
                                   "are about half of it); achieved and traffic are for the whole step on this rank, the unit the "
                                   "algorithmic bytes are defined on",
                         "kernel_ms": kern_ms, "alg_bytes_per_launch": ALG_BYTES_PER_COLUMN * ncol,
                         "kernels": kernels,
                         "kernels_note": "timing mode: kernels serialised with an event after each group, mean of 3 steps"},
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "diag": {"names": ["ppt_rain", "ppt_ice", "ppt_snow", "ppt_graupel", "lwp", "iwp", "active", "columns"],
                     "sum_over_steps": [float(x) for x in diag.tolist()]},
            "table_build_ms": th.table_build_ms,
        }
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            v, ms, init_s = cpu_reference_run(args.cpu_columns, 10, 1, cores)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "fortran_probe": fortran_probe(),
                                    "sample": "first %d columns of the bench domain x 10 steps (a rate), OpenMP over columns on %d "
                                              "threads; C++ restatement of the reference built -O3 without fast-math (no Fortran "
                                              "compiler on this box: see fortran_probe), init %.1f s excluded"
                                              % (args.cpu_columns, cores, init_s)}
        print(json.dumps(line), flush=True)
    th.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
