"""Which kernel serves a power-map call.

The kernel is chosen per call from the handle's kernel choice, its grid (a bflk_set_grid_fov grid, or caller tables with or
without bflk_set_grid_shape), the FIR setting and frame length, and the call's input: float rows (8-byte aligned, an even
number of samples apart, or not) or wire rows, one frame or many, synchronous or submitted.  An explicit choice that cannot
serve the call is refused with BFLK_ERR_STATE; the automatic choice falls back to the lane-broadcast kernel, then to the
generic one.  Every case runs on a fresh handle and reads kernel_info() after the call: the kernel it ran, whether the
register-tiled tables were built (tile span -1: never) and whether they fit (window chunks 0: they do not)."""
import numpy as np
import pytest

import cases

pytestmark = pytest.mark.gpu

H, W = 256, 1024
ROWS = COLS = 32   # 256 direction tiles: a few hundred frames fill the SMs with 16-warp CTAs
BFLK_ERR_STATE = -2
AUTO, GENERIC, TILED, BCAST, TILED_FMA2 = 0, 1, 2, 3, 4
STATE = "state"


def _fov_tables(N):
    w = _handle(N)
    w.set_grid_fov(ROWS, COLS, 180.0)
    off, fr = w.tables()
    w.close()
    return off, fr


def _handle(N):
    import bflk
    w = bflk.Beamformer(n_channels=64, frame_len=N, history=H, window_len=max(W, H + N + 1))
    w.set_tiled_geometry(cases.origins(1, 1))
    return w


def _route(kernel, grid="fov", wire=False, B=1, N=256, fir=False, odd=False, misaligned=False, submit=False):
    """kernel_info() after one call on a fresh handle, or STATE when the call is refused with BFLK_ERR_STATE."""
    import bflk
    import torch
    w = _handle(N)
    if grid == "fov":
        w.set_grid_fov(ROWS, COLS, 180.0)
    else:
        w.set_grid_tables(*_fov_tables(N))
        if grid == "tables+shape":
            w.set_grid_shape(ROWS, COLS)
    w.set_kernel(kernel)
    if fir:
        w.set_fir(np.full((16, 8), 1.0 / 8, np.float32))
    T = (B - 1) * N + W + (1 if odd else 0)
    power = torch.empty((B, w.n_directions()[2]), dtype=torch.float32, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(B)
    try:
        if wire:
            x = torch.randint(-(1 << 20), 1 << 20, (T, 64), dtype=torch.int32, device="cuda", generator=g)
            w.power_map_batch_i32_dev(x.data_ptr(), T, B, power.data_ptr())
        else:
            x = torch.randn(64 * T + 1, dtype=torch.float32, device="cuda", generator=g)
            ptr = x.data_ptr() + (4 if misaligned else 0)
            if submit:
                w.power_map_batch_dev_submit(ptr, T, B, power.data_ptr())
                w.power_map_batch_dev_join()
            else:
                w.power_map_batch_dev(ptr, T, B, power.data_ptr())
        torch.cuda.synchronize()
        assert torch.isfinite(power).all()
        return w.kernel_info()
    except bflk.BflkError as e:
        assert e.code == BFLK_ERR_STATE, e
        return STATE
    finally:
        torch.cuda.synchronize()
        w.close()


# (kernel, expected) of a call on a fov grid, and on caller tables with their grid shape declared: (kernel run, tables
# built, tables fit) or STATE
ON_A_GRID = [
    (AUTO, (TILED_FMA2, True, True)),
    (GENERIC, (GENERIC, False, False)),
    (TILED, (TILED, True, True)),
    (BCAST, (BCAST, False, False)),
    (TILED_FMA2, (TILED_FMA2, True, True)),
]
# caller tables without a grid shape: nothing to tile
WITHOUT_SHAPE = [
    (AUTO, (BCAST, True, False)),
    (GENERIC, (GENERIC, False, False)),
    (TILED, STATE),
    (BCAST, (BCAST, False, False)),
    (TILED_FMA2, STATE),
]
# float rows the tiled kernels cannot pack with 8-byte loads (odd row stride or misaligned start)
UNPACKABLE = [
    (AUTO, (BCAST, True, True)),
    (GENERIC, (GENERIC, False, False)),
    (TILED, STATE),
    (BCAST, (BCAST, False, False)),
    (TILED_FMA2, STATE),
]
# frame_len 128: too short for the tiled and the lane-broadcast kernels
SHORT_FRAMES = [
    (AUTO, (GENERIC, True, False)),
    (GENERIC, (GENERIC, False, False)),
    (TILED, STATE),
    (BCAST, STATE),
    (TILED_FMA2, STATE),
]


def _check(got, want):
    if want == STATE:
        assert got == STATE
        return
    assert got != STATE, "refused"
    last, span, nch = got
    assert (last, span >= 0, nch > 0) == want, got


@pytest.mark.parametrize("grid", ["fov", "tables+shape"])
@pytest.mark.parametrize("wire", [False, True], ids=["float", "wire"])
@pytest.mark.parametrize("kernel,want", ON_A_GRID)
def test_grid(kernel, want, grid, wire):
    _check(_route(kernel, grid, wire=wire), want)


@pytest.mark.parametrize("wire", [False, True], ids=["float", "wire"])
@pytest.mark.parametrize("kernel,want", WITHOUT_SHAPE)
def test_tables_without_shape(kernel, want, wire):
    _check(_route(kernel, "tables", wire=wire), want)


@pytest.mark.parametrize("kernel", [AUTO, GENERIC, TILED, BCAST, TILED_FMA2])
def test_tables_with_shape_route_as_the_fov_grid(kernel):
    """Declaring the shape of the fov grid's own tables gives the same kernel, tile span and window chunks."""
    assert _route(kernel, "tables+shape") == _route(kernel, "fov")


@pytest.mark.parametrize("how", ["odd_stride", "misaligned"])
@pytest.mark.parametrize("kernel,want", UNPACKABLE)
def test_unpackable_rows(kernel, want, how):
    _check(_route(kernel, odd=how == "odd_stride", misaligned=how == "misaligned"), want)


@pytest.mark.parametrize("kernel,want", [(AUTO, (GENERIC, False, False)), (GENERIC, (GENERIC, False, False)), (TILED, STATE)])
def test_fir(kernel, want):
    _check(_route(kernel, fir=True), want)


@pytest.mark.parametrize("kernel,want", SHORT_FRAMES)
def test_short_frames(kernel, want):
    _check(_route(kernel, N=128), want)


@pytest.mark.parametrize("kernel,grid,misaligned,want", [
    (AUTO, "fov", False, (TILED_FMA2, True, True)),
    (TILED, "fov", False, (TILED, True, True)),
    (AUTO, "fov", True, (BCAST, True, True)),          # falls back to a call on the caller's stream
    (TILED_FMA2, "fov", True, STATE),
    (GENERIC, "fov", False, (GENERIC, False, False)),
    (BCAST, "fov", False, (BCAST, False, False)),
    (AUTO, "tables", False, (BCAST, True, False)),
])
def test_submit(kernel, grid, misaligned, want):
    _check(_route(kernel, grid, misaligned=misaligned, submit=True), want)


@pytest.mark.parametrize("kernel", [AUTO, TILED])
def test_single_frame_then_batch(kernel):
    """A single frame runs in the latency CTA shape, a large batch in the throughput shape.  The shape is part of the
    tile tables, so the first call of each shape rebuilds them: three spread passes and one table pass, four launches."""
    import bflk
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = 1024
    assert bflk.launch_shape(ROWS, COLS, 64, n_frames=1, n_sms=sms)[0] > 0
    assert bflk.launch_shape(ROWS, COLS, 64, n_frames=B, n_sms=sms)[0] == 0
    w = _handle(256)
    w.set_grid_fov(ROWS, COLS, 180.0)
    w.set_kernel(kernel)
    want = TILED_FMA2 if kernel == AUTO else TILED
    x = torch.randn((64, (B - 1) * 256 + W), dtype=torch.float32, device="cuda")
    power = torch.empty((B, ROWS * COLS), dtype=torch.float32, device="cuda")
    spent = []
    for n in (1, 1, B, B, 1):
        before = w.launch_count()
        w.power_map_batch_dev(x.data_ptr(), x.shape[1], n, power.data_ptr())
        spent.append(w.launch_count() - before)
        assert w.kernel_info()[0] == want
    torch.cuda.synchronize()
    assert spent[0] - spent[1] == 4 and spent[2] - spent[3] == 4 and spent[4] == spent[0], spent
    w.close()
