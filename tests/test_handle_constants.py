"""Two handles on one device whose scheme constants differ (set_Nc 100 and 3000, both mixed-phase with sedimentation) step at
the same time from two threads, each on its own stream, through kidmp_step_device and the device WRF tile entry.  Every
kernel gets its handle's constants with its launch, so each handle computes, bit for bit, what it computes alone."""
import threading

import numpy as np
import pytest

import regimes as R
from parity_util import FIELDS

NI, NJ = 256, 128                        # 32 768 bench-like columns, also stepped as one WRF tile of NI x 60 x NJ
DT = 60.0                                # with dz = 100 m: columns with sedimentation sub-steps
STEPS = 3                                # kidmp_step_device calls of one round, then one device tile call
ROUNDS = 2                               # rounds of each thread in the concurrent run
SET_NC = (100.0, 3000.0)


class Run:
    """One handle, its torch stream and device copies of its inputs, allocated once.  round() starts from the inputs, takes
    STEPS chained steps and one WRF tile step, and returns every output and the handle's diagnostics of the round."""

    def __init__(self, set_Nc, st, p, dz):
        import torch
        from kid_b200.kidmp import Thompson
        self.th = Thompson(set_Nc=set_Nc, iiwarm=False, l_sediment=True)
        self.s = torch.cuda.Stream()
        nz = self.nz = dz.shape[0]
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()
        self.src = {k: dev(st[k]) for k in FIELDS}
        self.f = {k: v.clone() for k, v in self.src.items()}
        self.p, self.dz = dev(p), dev(dz)
        self.ppt = torch.zeros((4, NI * NJ), dtype=torch.float32, device="cuda")
        to3 = lambda a: np.ascontiguousarray(a.reshape(nz, NJ, NI).transpose(1, 0, 2))      # [k][col] -> (nj, nk, ni)
        p3 = to3(p)
        pii = ((p3 / 1.0e5) ** (287.04 / 1004.0)).astype(np.float32)
        src3 = {k: to3(st[k]) for k in FIELDS if k != "t"}
        src3["th"] = (to3(st["t"]) / pii).astype(np.float32)
        self.src3 = {k: dev(v) for k, v in src3.items()}
        self.f3 = {k: v.clone() for k, v in self.src3.items()}
        self.pii, self.p3 = dev(pii), dev(p3)
        self.dz3 = dev(np.broadcast_to(dz.reshape(1, nz, 1), (NJ, nz, NI)))
        self.acc = {k: torch.zeros((NJ, NI), dtype=torch.float32, device="cuda")
                    for k in ("rainnc", "rainncv", "sr", "snownc", "snowncv", "graupelnc", "graupelncv")}
        self.radii = {k: torch.zeros((NJ, nz, NI), dtype=torch.float32, device="cuda") for k in ("re_cloud", "re_ice", "re_snow")}
        torch.cuda.synchronize()

    def round(self):
        import torch
        self.th.diag()                                   # (clears the domain sums)
        with torch.cuda.stream(self.s):
            for k in self.f:
                self.f[k].copy_(self.src[k])
            for k in self.f3:
                self.f3[k].copy_(self.src3[k])
            for a in list(self.acc.values()) + list(self.radii.values()):
                a.zero_()
        for _ in range(STEPS):
            self.th.step_device(NI * NJ, self.nz, DT, [self.f[k].data_ptr() for k in FIELDS], self.p.data_ptr(),
                                self.dz.data_ptr(), self.ppt.data_ptr(), stream=self.s.cuda_stream)
        self.th.mp_gt_driver_device(DT, self.f3, self.pii, self.p3, self.dz3, self.acc, radii=self.radii, stream=self.s)
        self.s.synchronize()
        out = {"state_" + k: v.cpu().numpy() for k, v in self.f.items()}
        for k, v in list(self.f3.items()) + list(self.acc.items()) + list(self.radii.items()):
            out["wrf_" + k] = v.cpu().numpy()
        out["ppt"] = self.ppt.cpu().numpy()
        out["diag"] = self.th.diag()
        return out

    def close(self):
        self.th.close()


def _same_bits(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def _mismatches(got, ref):
    return [k for k in ref if not _same_bits(got[k], ref[k])]


@pytest.fixture(scope="module")
def runs():
    st, p, dz = R.bench_like(NI * NJ, 100.0)
    rs = [Run(n, st, p, dz) for n in SET_NC]
    yield rs
    for r in rs:
        r.close()


@pytest.mark.gpu
def test_two_handles_with_different_constants_at_once(runs):
    refs = [r.round() for r in runs]                    # each handle alone
    # the handles' results differ where the constants do (set_Nc: droplet number, radii), so a swap would show
    assert _mismatches(refs[0], refs[1]), "both handles computed the same numbers"
    assert not _mismatches(runs[0].round(), refs[0]), "a second solo round differs from the first"
    got = [[] for _ in runs]
    errors = []
    barrier = threading.Barrier(len(runs))

    def work(i):
        try:
            barrier.wait()
            for _ in range(ROUNDS):
                got[i].append(runs[i].round())
        except Exception as e:                           # (reported below: an assertion in a thread would be lost)
            errors.append(e)
    threads = [threading.Thread(target=work, args=(i,)) for i in range(len(runs))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for i, n in enumerate(SET_NC):
        for j, g in enumerate(got[i]):
            bad = _mismatches(g, refs[i])
            assert not bad, "set_Nc %g, round %d: %s differ from the solo run" % (n, j, bad)
