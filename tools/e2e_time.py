"""End-to-end time of kidmp_step with pinned host arrays (H2D + kernels + D2H every step), the path bench.py reports as e2e.
    KIDMP_PIPE_CHUNK=131072 python tools/e2e_time.py [--columns N] [--steps K] [--aero] [--gpus N]
--aero: kidmp_step_aero (is_aerosol_aware = .true.) on the same pinned state with pinned nc, nwfa, nifa, w and nwfa2d, steps
alternating with the plain kidmp_step; both times are printed.  --gpus N: one handle over N GPUs (kidmp_config::ndev).
KIDMP_PIPE_TRACE=1 prints the device timeline of every chunk on stderr."""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from kid_b200 import synth  # noqa: E402
from kid_b200.kidmp import Thompson, FIELDS  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--columns", type=int, default=1048576)
ap.add_argument("--steps", type=int, default=5)
ap.add_argument("--aero", action="store_true")
ap.add_argument("--gpus", type=int, default=1)
a = ap.parse_args()
if a.gpus > torch.cuda.device_count():
    sys.exit("--gpus %d: this box has %d" % (a.gpus, torch.cuda.device_count()))
try:
    limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30).stdout.strip() or "unknown"
except Exception:
    limit = "unknown"
print("card", torch.cuda.get_device_name(0), "power limit", limit, "gpus", a.gpus)
th = Thompson(set_Nc=100.0, iiwarm=False, l_sediment=True, devices=list(range(a.gpus)) if a.gpus > 1 else None)
st, p, dz = synth.make_domain(a.columns, nz=60, nx=1024, device="cuda")
pinned = lambda x: torch.as_tensor(x).to("cpu").pin_memory()
host = {k: pinned(st[k]) for k in FIELDS}
hp = pinned(p)
hs = {k: host[k].numpy() for k in FIELDS}
hpn, hdz = hp.numpy(), dz.cpu().numpy()
if a.aero:
    nc, nwfa, nifa, w = synth.make_aerosols(host, hp)
    ae = {k: pinned(v) for k, v in (("nc", nc), ("nwfa", nwfa), ("nifa", nifa))}
    aen = {k: v.numpy() for k, v in ae.items()}
    hw = pinned(w).numpy()
    hn2 = pinned(torch.empty(a.columns).uniform_(0.0, 1.0e5, generator=torch.Generator().manual_seed(5))).numpy()
    del nc, nwfa, nifa, w
del st, p


def timed(fn):
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e3


plain = lambda: th.step(10.0, hs, hpn, hdz)
aero = lambda: th.step_aero(10.0, hs, aen, hpn, hw, hdz, nwfa2d=hn2)
plain()
if a.aero:
    aero()
ms, ms_aero = [], []
for _ in range(a.steps):
    ms.append(timed(plain))
    if a.aero:
        ms_aero.append(timed(aero))
cells = a.columns * 60 * 4 / 1e9
tag = "pipe_chunk %s zerocopy %s" % (os.environ.get("KIDMP_PIPE_CHUNK", "default"), os.environ.get("KIDMP_ZEROCOPY", "1"))
print(tag, "plain ms", " ".join("%.1f" % x for x in ms), "H2D %.2f GB, %.1f GB/s" % (10 * cells, 10 * cells / (min(ms) * 1e-3)))
if a.aero:
    gb = 14 * cells + a.columns * 4 / 1e9                  # nine fields, p, nc, nwfa, nifa, w and nwfa2d
    print(tag, "aero ms", " ".join("%.1f" % x for x in ms_aero), "H2D %.2f GB, %.1f GB/s" % (gb, gb / (min(ms_aero) * 1e-3)),
          "zero_copy_return", th.step_stats()["zero_copy_return"])
th.close()
