"""What a handle keeps between calls and what it gives back when it is destroyed.

bflk_targets and bflk_heatmap with a NULL map read the map the last single-frame host batch left on the device: no other
call may overwrite it, and a batch of several frames leaves none.  Creating a handle, using every kind of call on it and
destroying it again must return all of its device memory, for a lone handle and for the handles of a group."""
import ctypes as C

import numpy as np
import pytest

import cases

pytestmark = pytest.mark.gpu

N, W = 256, 1024
BFLK_ERR_STATE = -2


def _heatmap(w, power=None):
    """bflk_heatmap; power None: the map left on the device"""
    n = w.n_directions()[2]
    heat = np.zeros(n, np.uint8)
    arg, mx = C.c_int32(), C.c_float()
    src = None if power is None else np.ascontiguousarray(power, np.float32)
    w._check(w._L.bflk_heatmap(w._h, None if src is None else src.ctypes.data, n, heat.ctypes.data, C.byref(arg), C.byref(mx)))
    return heat, arg.value, mx.value


def _targets(w, power=None, max_targets=16, min_rel_power=0.05):
    """bflk_targets; power None: the map left on the device"""
    import bflk
    out = (bflk.Target * max_targets)()
    n = C.c_int32()
    src = None if power is None else np.ascontiguousarray(power, np.float32)
    w._check(w._L.bflk_targets(w._h, None if src is None else src.ctypes.data, max_targets, min_rel_power, out, C.byref(n)))
    return [(t.direction, t.power, t.probability) for t in out[:n.value]]


def _window():
    from bflk import synth
    return synth.make_stream(synth.tile_geometry(cases.origins(1, 1)), W)


def _assert_device_map_is(w, p):
    got_t, got_h = _targets(w), _heatmap(w)
    assert got_t == _targets(w, p)
    heat, arg, mx = _heatmap(w, p)
    assert np.array_equal(got_h[0], heat) and got_h[1:] == (arg, mx)


@pytest.mark.parametrize("between", ["heatmap", "fp32_peak_tflops", "calibrate"])
def test_other_calls_leave_the_map_on_the_device(between):
    import bflk
    w = bflk.MIMOWorker(cases.origins(1, 1), 16, 16, 180.0)
    window = _window()
    p = w.power_map(window)
    if between == "heatmap":
        w.heatmap(np.linspace(1.0, 2.0, p.size, dtype=np.float32)[::-1].copy())   # another host map of the same size
    elif between == "fp32_peak_tflops":
        assert w.fp32_peak_tflops() > 0
    else:
        w.calibrate(window)                                                        # 64 channel powers
    _assert_device_map_is(w, p)


def test_single_frame_wire_map_stays_on_the_device():
    import bflk
    w = bflk.MIMOWorker(cases.origins(1, 1), 16, 16, 180.0)
    frames = np.random.default_rng(5).integers(-(1 << 20), 1 << 20, (W, 64), dtype=np.int32)
    p = w.power_map_i32(frames)
    _assert_device_map_is(w, p)


def test_multi_frame_wire_batch_leaves_no_map():
    import bflk
    w = bflk.MIMOWorker(cases.origins(1, 1), 16, 16, 180.0)
    w.power_map(_window())
    B = 4
    frames = np.random.default_rng(6).integers(-(1 << 20), 1 << 20, ((B - 1) * N + W, 64), dtype=np.int32)
    w.power_map_batch_i32(frames, B)
    with pytest.raises(bflk.BflkError) as e:
        _targets(w)
    assert e.value.code == BFLK_ERR_STATE


# ---- nothing leaks -----------------------------------------------------------------------------------------------------
B_LEAK = 592          # a cfg3 batch as bench.py runs it: 512 channels x 152 320 samples = 312 MB per copy of the input
CYCLES = 3
# Free device memory after every cycle must come back to within this of its value after the first one.  A cycle allocates
# well over 1 GiB (the float batch's window, two asynchronous input buffers, the wire samples, the kernels' scratch), so a
# lost buffer shows.  The tolerance is not derived from a measurement; it only has to stay below the smallest of them.
TOLERANCE = 64 << 20


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _group_handle(group, i):
    """Handle i of a group, with the Beamformer methods; the group owns and destroys it."""
    import bflk

    class Borrowed(bflk.Beamformer):
        def __init__(self):
            self._L, self.cfg = group._L, group.cfg
            self._h = C.c_void_p(group._L.bflk_group_handle(group._g, i))

        def close(self):
            pass

    return Borrowed()


class _Inputs:
    """The inputs of one cycle, allocated once so that torch's caching allocator holds the same memory every cycle."""

    def __init__(self, devices):
        import torch
        from bflk import synth
        c = cases.CONFIGS["cfg3"]
        xyz = synth.tile_geometry(cases.origins(c["nx"], c["ny"]))
        T = (B_LEAK - 1) * N + W
        self.T = T
        stream = synth.make_stream(xyz, T)
        self.stream = torch.from_numpy(stream).pin_memory()
        self.out = torch.zeros((2, B_LEAK, c["rows"] * c["cols"]), dtype=torch.float32).pin_memory()
        self.wire = np.ascontiguousarray(stream.T).view(np.int32) >> 8
        self.window = np.ascontiguousarray(stream[:, :W])
        self.dev_in = {d: torch.from_numpy(stream).to(f"cuda:{d}") for d in devices}
        self.dev_out = {d: torch.zeros((B_LEAK, c["rows"] * c["cols"]), dtype=torch.float32, device=f"cuda:{d}") for d in devices}
        self.theta, self.phi = cases.cfg4_targets()


def _use(h, device, x):
    """Every kind of call a handle serves, with timing on and its event pairs never collected."""
    import torch
    h.enable_timing(True)
    h.power_map_batch_ptr(x.stream.data_ptr(), x.T, B_LEAK, x.out[0].data_ptr())
    for k in range(2):
        h.power_map_batch_submit_ptr(x.stream.data_ptr(), x.T, B_LEAK, x.out[k].data_ptr())
    for k in range(2):
        h.power_map_batch_wait()
    h.power_map_batch_dev_submit(x.dev_in[device].data_ptr(), x.T, B_LEAK, x.dev_out[device].data_ptr())
    h.power_map_batch_dev_join()
    torch.cuda.synchronize(device)
    h.power_map_batch_i32(x.wire, B_LEAK)
    h.miso(x.theta, x.phi, x.window)
    h.monopulse(x.theta, x.phi, x.window, spread=0.05, theta_limit=1.2)


def _free(devices):
    import torch
    for d in devices:
        torch.cuda.synchronize(d)
    return [torch.cuda.mem_get_info(d)[0] for d in devices]


def _check_cycles(devices, cycle):
    x = _Inputs(devices)
    after = []
    for _ in range(CYCLES):
        before = _free(devices)
        used = cycle(x)            # free memory while the handles still exist
        assert max(b - u for b, u in zip(before, used)) > 1 << 30, "the cycle must allocate over 1 GiB"
        after.append(_free(devices))
    drift = [max(a0 - a for a0, a in zip(after[0], a1)) for a1 in after[1:]]
    print(f"free memory lost after cycles 2..{CYCLES} relative to cycle 1, per device maximum: {drift} bytes")
    assert all(d <= TOLERANCE for d in drift), drift


def test_handle_returns_its_memory():
    import bflk
    c = cases.CONFIGS["cfg3"]

    def cycle(x):
        w = bflk.MIMOWorker(cases.origins(c["nx"], c["ny"]), c["rows"], c["cols"], c["fov"])
        _use(w, 0, x)
        used = _free([0])
        w.close()
        return used

    _check_cycles([0], cycle)


@pytest.mark.parametrize("n_devices", [1, 2])
def test_group_returns_its_memory(n_devices):
    import bflk
    if _n_gpus() < n_devices:
        pytest.skip(f"needs {n_devices} GPUs in one box")
    c = cases.CONFIGS["cfg3"]
    devices = list(range(n_devices))

    def cycle(x):
        g = bflk.Group(cases.origins(c["nx"], c["ny"]), c["rows"], c["cols"], c["fov"], devices=devices)
        g.power_map_batch(x.stream.numpy(), B_LEAK)
        g.power_map_batch_dev([x.dev_in[d].data_ptr() for d in devices], x.T, B_LEAK, [x.dev_out[d].data_ptr() for d in devices])
        for i, d in enumerate(devices):
            _use(_group_handle(g, i), d, x)
        used = _free(devices)
        g.close()
        return used

    _check_cycles(devices, cycle)
