"""Per-call time of the WRF / MPAS entries on a WRF-sized patch, and what the tile gather / scatter costs.

Memory box 210 x 51 x 210 (ims:ime, kms:kme, jms:jme): a 5-point halo on all four sides and one spare level on top
(kme = kte + 1) around a tile of 200 x 50 x 200 columns x levels.  Four figures, median of --calls calls each after --warmup:

  packed       kidmp_mp_gt_driver on the tile packed into arrays of its own (host arrays; what a host has to do today
               after packing the tile itself - that packing is not counted)
  tile_host    kidmp_mp_gt_driver_tile on the memory box (host arrays; the library stages the tile rows)
  tile_device  kidmp_mp_gt_driver_tile_device on the memory box as CUDA tensors (device events around the call)
  step_device  kidmp_step_device on the same columns already in [k][col] planes (device events): tile_device minus this is
               the gather, scatter and accumulators of the device entry

Every call starts from the same inputs (restored outside the timed region), so every call does the same work.  The layer
depths are the same in every column, so that kidmp_step_device (one shared dz vector) steps exactly what the WRF entries
step.  Host times are wall time of a call that returns synchronised.  Prints the GPU's name and power limit, then one JSON
line.

    python tools/wrf_tile_time.py [--calls 20] [--warmup 3] [--out result.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

F3 = ("qv", "qc", "qr", "qi", "qs", "qg", "ni", "nr", "th")
ACC = ("rainnc", "rainncv", "sr", "snownc", "snowncv", "graupelnc", "graupelncv")


def tile_case(ni, nk, nj, seed=3):
    """(nj, nk, ni) arrays of one tile from the synthetic cloudy domain, theta + Exner function, accumulators with a history."""
    from kid_b200 import synth
    rng = np.random.default_rng(seed)
    st, p, dz = synth.make_domain(ni * nj, nz=nk, coherent=False, cloudy_fraction=0.6)
    st = {k: v.numpy() for k, v in st.items()}
    to3 = lambda a: np.ascontiguousarray(a.reshape(nk, nj, ni).transpose(1, 0, 2))
    v = {k: to3(st[k]) for k in ("qv", "qc", "qr", "qi", "qs", "qg", "ni", "nr")}
    v["p"] = to3(p.numpy())
    v["pii"] = ((v["p"] / 1.0e5) ** (287.04 / 1004.0)).astype(np.float32)
    v["th"] = (to3(st["t"]) / v["pii"]).astype(np.float32)
    v["dz"] = np.ascontiguousarray(np.broadcast_to(dz.numpy().reshape(1, nk, 1), (nj, nk, ni))).astype(np.float32)
    for k in ACC:
        v[k] = (rng.random((nj, ni)) * 3.0).astype(np.float32)
    for k in ("re_cloud", "re_ice", "re_snow"):
        v[k] = np.zeros((nj, nk, ni), np.float32)
    return v, dz.numpy()


def embed(v, mem_shape, s3):
    out = {}
    for k, a in v.items():
        m = np.zeros(mem_shape if a.ndim == 3 else (mem_shape[0], mem_shape[2]), np.float32)
        m[s3 if a.ndim == 3 else (s3[0], s3[2])] = a
        out[k] = m
    return out


def gpu_identity():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                       # (the figure is then reported as unknown, never guessed)
        pl = "unknown (%s)" % e
    return name, pl


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--halo", type=int, default=5)
    ap.add_argument("--tile", type=int, nargs=3, default=(200, 50, 200), metavar=("NI", "NK", "NJ"))
    ap.add_argument("--out")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("wrf_tile_time.py: no CUDA device")
    from kid_b200.kidmp import Thompson, WrfTile, FIELDS
    ni, nk, nj = args.tile
    hw = args.halo
    mem_shape = (nj + 2 * hw, nk + 1, ni + 2 * hw)
    s3 = (slice(hw, hw + nj), slice(0, nk), slice(hw, hw + ni))
    tile = WrfTile(hw, ni, 0, nk, hw, nj)
    v, dzv = tile_case(ni, nk, nj)
    mem = embed(v, mem_shape, s3)
    th = Thompson(set_Nc=100.0, iiwarm=False, l_sediment=True)
    L, h, dt = th._L, th.h, 20.0
    host_ptr = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
    dev_ptr = lambda a: C.cast(C.c_void_p(int(a.data_ptr())), C.POINTER(C.c_float))

    def structs(arrs, addr):
        f3 = {k: arrs[k] for k in F3}
        return th._wrf_structs(f3, arrs["pii"], arrs["p"], arrs["dz"], {k: arrs[k] for k in ACC},
                               {k: arrs[k] for k in ("re_cloud", "re_ice", "re_snow")}, None, arrs["qv"].shape, addr)

    def host_timer(arrs, pristine, call):
        ts = []
        for it in range(args.warmup + args.calls):
            for k in arrs:
                np.copyto(arrs[k], pristine[k])
            t0 = time.perf_counter()
            rc = call()
            t1 = time.perf_counter()
            if rc:
                raise RuntimeError(L.kidmp_last_error(h).decode())
            if it >= args.warmup:
                ts.append((t1 - t0) * 1e3)
        return float(np.median(ts)), ts

    def dev_timer(arrs, pristine, call, stream):
        pairs = []
        with torch.cuda.stream(stream):
            for it in range(args.warmup + args.calls):
                for k in arrs:
                    arrs[k].copy_(pristine[k])
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                rc = call()
                e1.record(stream)
                if rc:
                    raise RuntimeError(L.kidmp_last_error(h).decode())
                if it >= args.warmup:
                    pairs.append((e0, e1))
        stream.synchronize()
        ts = [a.elapsed_time(b) for a, b in pairs]
        return float(np.median(ts)), ts

    res = {}
    # 1. packed entry on the pre-packed tile
    packed = {k: a.copy() for k, a in v.items()}
    w1, _, _, keep1 = structs(packed, host_ptr)
    res["packed_ms"], _ = host_timer(packed, v, lambda: L.kidmp_mp_gt_driver(h, C.byref(w1), dt))
    # 2. tile host entry on the memory box
    memw = {k: a.copy() for k, a in mem.items()}
    w2, _, _, keep2 = structs(memw, host_ptr)
    res["tile_host_ms"], _ = host_timer(memw, mem, lambda: L.kidmp_mp_gt_driver_tile(h, C.byref(w2), C.byref(tile), None, dt))
    same = all(np.array_equal(memw[k][s3 if memw[k].ndim == 3 else (s3[0], s3[2])], packed[k]) for k in packed)
    # 3. tile device entry on the memory box
    s = torch.cuda.Stream()
    dmem0 = {k: torch.from_numpy(a).cuda() for k, a in mem.items()}
    dmem = {k: a.clone() for k, a in dmem0.items()}
    w3, _, _, keep3 = structs(dmem, dev_ptr)
    torch.cuda.synchronize()
    res["tile_device_ms"], _ = dev_timer(dmem, dmem0, lambda: L.kidmp_mp_gt_driver_tile_device(
        h, C.byref(w3), C.byref(tile), None, dt, C.c_void_p(s.cuda_stream)), s)
    same = same and all(np.array_equal(dmem[k].cpu().numpy(), memw[k]) for k in memw)
    # 4. kidmp_step_device on the same columns in [k][col] planes
    planes = lambda a: np.ascontiguousarray(a.transpose(1, 0, 2).reshape(nk, nj * ni))
    st0 = {k: torch.from_numpy(planes(v[k])).cuda() for k in ("qv", "qc", "qi", "qr", "qs", "qg", "ni", "nr")}
    st0["t"] = torch.from_numpy(planes(v["th"] * v["pii"])).cuda()
    st = {k: a.clone() for k, a in st0.items()}
    dp = torch.from_numpy(planes(v["p"])).cuda()
    ddz = torch.from_numpy(np.ascontiguousarray(dzv)).cuda()
    dppt = torch.zeros((4, ni * nj), dtype=torch.float32, device="cuda")
    fp = (C.c_void_p * 9)(*[C.c_void_p(st[k].data_ptr()) for k in FIELDS])
    torch.cuda.synchronize()
    res["step_device_ms"], _ = dev_timer(st, st0, lambda: L.kidmp_step_device(
        h, ni * nj, nk, dt, fp, C.c_void_p(dp.data_ptr()), C.c_void_p(ddz.data_ptr()), C.c_void_p(dppt.data_ptr()),
        C.c_void_p(s.cuda_stream)), s)
    same_step = all(np.array_equal(st[k].cpu().numpy(), planes(packed[k])) for k in ("qv", "qc", "qi", "qr", "qs", "qg", "ni", "nr"))
    th.close()
    name, pl = gpu_identity()
    res.update(gpu=name, power_limit=pl, memory_box=list(mem_shape[::-1]), tile=list(args.tile), halo=hw,
               calls=args.calls, warmup=args.warmup, tile_equals_packed=bool(same), step_device_equals_packed=bool(same_step),
               gather_scatter_ms=res["tile_device_ms"] - res["step_device_ms"],
               host_tile_over_packed_ms=res["tile_host_ms"] - res["packed_ms"])
    print("GPU %s, power limit %s" % (name, pl))
    print("memory box %d x %d x %d (i, k, j), tile %d x %d x %d, median of %d calls" % (
        mem_shape[2], mem_shape[1], mem_shape[0], ni, nk, nj, args.calls))
    for k in ("packed_ms", "tile_host_ms", "tile_device_ms", "step_device_ms"):
        print("  %-16s %8.3f ms" % (k[:-3], res[k]))
    print(json.dumps(res), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
