"""A step runs on one work set, on the caller's stream: the removed scheduling options are refused, a handle waits for its own
work rather than the whole device (so its first step may run while another thread captures a CUDA graph), and a host-pipeline
chunk is never larger than a launch chunk (so the column flags of the chunk are those of its one launch)."""
import threading

import numpy as np
import pytest

from parity_util import FIELDS

pytestmark = pytest.mark.gpu

CFG = dict(set_Nc=100.0, iiwarm=False, l_sediment=True)
NZ = 60
REMOVED = ("lanes", "lane_min", "stagger", "cell_blocks", "l2_window", "fuse", "units")
KEPT = {"chunk": 1 << 20, "timing": 0, "graphs": 1, "simple": 1, "classes": 1}        # (their defaults)


@pytest.fixture(scope="module")
def reference():
    """A handle with default options, made before any test of this module changes the environment."""
    from kid_b200.kidmp import Thompson
    th = Thompson(**CFG)
    yield th
    th.close()


def _device_domain(ncol, col0):
    import torch
    from kid_b200 import synth
    st, p, dz = synth.make_domain(ncol, nz=NZ, col0=col0, nx=1024, cloudy_fraction=0.7, coherent=False, device="cuda")
    return st, p, dz, torch.zeros((4, ncol), dtype=torch.float32, device="cuda")


def _step_device(th, st, p, dz, ppt, dt=10.0):
    th.step_device(ppt.shape[1], NZ, dt, [st[k].data_ptr() for k in FIELDS], p.data_ptr(), dz.data_ptr(), ppt.data_ptr())
    th.sync()


def _assert_same_bits(got, want, what):
    for k in FIELDS:
        assert np.array_equal(got[k].view(np.uint32), want[k].view(np.uint32)), (what, k)


def test_removed_options_are_refused(reference):
    """Each removed option gets the unknown-option error, and the handle still steps as a fresh one does."""
    import torch
    from kid_b200.kidmp import KidmpError, Thompson
    st, p, dz, ppt = _device_domain(5000, 310000)
    th = Thompson(**CFG)
    try:
        for name in REMOVED:
            with pytest.raises(KidmpError, match="unknown option"):
                th.set_option(name, 1)
        got, got_ppt = {k: v.clone() for k, v in st.items()}, ppt.clone()
        _step_device(th, got, p, dz, got_ppt)
        want, want_ppt = {k: v.clone() for k, v in st.items()}, ppt.clone()
        _step_device(reference, want, p, dz, want_ppt)
        torch.cuda.synchronize()
        _assert_same_bits({k: v.cpu().numpy() for k, v in got.items()}, {k: v.cpu().numpy() for k, v in want.items()}, "state")
        assert np.array_equal(got_ppt.cpu().numpy().view(np.uint32), want_ppt.cpu().numpy().view(np.uint32))
        assert want_ppt.abs().sum() > 0
        for name, value in KEPT.items():
            th.set_option(name, value)
    finally:
        th.close()


def test_first_step_while_another_thread_captures(reference):
    """Thread A captures a torch op into a CUDA graph on a side stream (relaxed mode).  While that capture is open, thread B runs
    the first step of a fresh handle, which allocates its work buffers: the handle waits for its own earlier work only, so
    B's step succeeds with the bits of a step outside any capture, and A's capture ends cleanly and replays."""
    import torch
    from kid_b200.kidmp import Thompson
    st, p, dz, ppt = _device_domain(3000, 320000)
    got, got_ppt = {k: v.clone() for k, v in st.items()}, ppt.clone()
    want, want_ppt = {k: v.clone() for k, v in st.items()}, ppt.clone()
    _step_device(reference, want, p, dz, want_ppt)
    x = torch.arange(4096, dtype=torch.float32, device="cuda")
    y = torch.zeros_like(x)
    side = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    torch.cuda.synchronize()
    made, capturing, stepped = threading.Event(), threading.Event(), threading.Event()
    errors, handles = [], []

    def capture():                                   # thread A
        try:
            assert made.wait(600)
            with torch.cuda.graph(g, stream=side, capture_error_mode="relaxed"):
                torch.mul(x, 2.0, out=y)
                capturing.set()
                assert stepped.wait(600)
        except BaseException as e:                   # (reported below: an assertion in a thread would be lost)
            errors.append(("capture", e))
        finally:
            capturing.set()

    def first_step():                                # thread B
        try:
            # (the handle is made before the capture opens: its init frees the scratch of the table build, and whether a
            # cudaFree is safe during another thread's capture is not what this test is about)
            th = Thompson(**CFG)
            handles.append(th)
            made.set()
            assert capturing.wait(600)
            _step_device(th, got, p, dz, got_ppt)
        except BaseException as e:
            errors.append(("step", e))
        finally:
            made.set()
            stepped.set()
    threads = [threading.Thread(target=capture), threading.Thread(target=first_step)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    try:
        assert not errors, errors
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(y, x * 2.0)
        _assert_same_bits({k: v.cpu().numpy() for k, v in got.items()}, {k: v.cpu().numpy() for k, v in want.items()}, "state")
        assert np.array_equal(got_ppt.cpu().numpy().view(np.uint32), want_ppt.cpu().numpy().view(np.uint32))
    finally:
        for th in handles:
            th.close()


def test_pipelined_step_with_launch_chunk_below_pipeline_chunk(reference, monkeypatch):
    """kidmp_step on pinned column-fastest arrays with "chunk" (columns per launch) below KIDMP_PIPE_CHUNK: the pipeline
    chunk shrinks to the launch chunk, so the changed columns k_scatter_host writes back are those of the chunk's own launch.
    Same bits as the default handle over three steps."""
    from kid_b200 import synth
    from kid_b200.kidmp import Thompson
    ncol = 3 * 4096 + 77
    st, p, dz = synth.make_domain(ncol, nz=NZ, col0=330000, nx=1024, cloudy_fraction=0.6, coherent=False)
    want = {k: v.numpy().copy() for k, v in st.items()}
    monkeypatch.setenv("KIDMP_PIPE_CHUNK", "4096")
    th = Thompson(**CFG)
    try:
        th.set_option("chunk", 1024)
        pinned = {k: v.clone().pin_memory() for k, v in st.items()}
        got = {k: v.numpy() for k, v in pinned.items()}
        for step in range(3):
            ppt_want = reference.step(10.0, want, p.numpy().copy(), dz.numpy())
            ppt_got = th.step(10.0, got, p.numpy().copy(), dz.numpy())
            assert th.step_stats()["zero_copy_return"] == 1, step
            _assert_same_bits(got, want, "step %d" % step)
            assert np.array_equal(ppt_got.view(np.uint32), ppt_want.view(np.uint32)), step
        assert not np.array_equal(want["qc"], st["qc"].numpy())
        assert ppt_want.any()
    finally:
        th.close()
