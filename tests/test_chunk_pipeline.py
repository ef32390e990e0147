"""Chunked host batches at a small chunk size (BFLK_CHUNK_MIB=1): batches of a few hundred kilobytes per chunk travel in
several chunks whose kernels alternate between the handle's two compute streams, so the chunk pipeline runs for every
kernel, input format and option on small inputs.  Every frame must come out with the bits of the same frame computed in a
small batch that fits one chunk."""
import numpy as np
import pytest

import cases

pytestmark = pytest.mark.gpu

B = 160          # 64 channels x 160 frames x 1 KiB = 10 MiB: several 1-MiB chunks (at least three for the tiled kernels)
SMALL = 10       # frames per reference batch: one chunk
N, W = 256, 1024


@pytest.fixture
def bf(monkeypatch):
    monkeypatch.setenv("BFLK_CHUNK_MIB", "1")      # read by bflk_create: set before every handle
    import bflk
    return bflk


def _stream(n_frames):
    from bflk import synth
    base = synth.make_stream(synth.tile_geometry(cases.origins(1, 1)), 40 * N + W)
    s = np.ascontiguousarray(np.tile(base[:, :40 * N], (1, n_frames // 40 + 2))[:, :(n_frames - 1) * N + W])
    s *= np.linspace(0.5, 1.5, s.shape[1], dtype=np.float32)[None, :]                # no two frames alike
    return s


def _worker(bf, kernel, variant, golden):
    w = bf.MIMOWorker(cases.origins(1, 1), 16, 16, 180.0)
    w.set_kernel(kernel)
    if variant == "range":
        w.set_direction_range(37, 150)
    elif variant == "fir":
        w.set_fir(golden["fir"]["coeffs"])
    return w


def _batch(w, source, data, n_frames):
    if source == "wire":
        return w.power_map_batch_i32(data, n_frames)
    if source == "pageable":
        return w.power_map_batch(data, n_frames)
    import torch
    t = torch.from_numpy(data).pin_memory()
    out = torch.zeros((n_frames, w.n_directions()[2]), dtype=torch.float32).pin_memory()
    w.power_map_batch_ptr(t.data_ptr(), data.shape[1], n_frames, out.data_ptr())
    return out.numpy().copy()


def _frames(source, data, b0, nb):
    if source == "wire":
        return np.ascontiguousarray(data[b0 * N:(b0 + nb - 1) * N + W])
    return np.ascontiguousarray(data[:, b0 * N:(b0 + nb - 1) * N + W])


CASES = [(k, v) for v in ("plain", "range") for k in (0, 1, 2, 3)] + [(0, "fir"), (1, "fir")]


@pytest.mark.parametrize("source", ["pinned", "pageable", "wire"])
@pytest.mark.parametrize("kernel,variant", CASES)
def test_chunked_batch_equals_single_chunk_batches(bf, golden, source, kernel, variant):
    from bflk import synth
    w = _worker(bf, kernel, variant, golden)
    stream = _stream(B)
    data = synth.to_wire_i32(stream) if source == "wire" else stream
    full = _batch(w, source, data, B)
    assert np.all(np.isfinite(full)) and full.min() > 0
    if kernel:
        assert w.kernel_info()[0] == kernel
    elif variant == "fir":
        assert w.kernel_info()[0] == 1                   # FIR interpolation runs through the generic kernel
    for b0 in range(0, B, SMALL):                          # every frame, so every chunk boundary
        part = _batch(w, source, _frames(source, data, b0, SMALL), SMALL)
        assert np.array_equal(full[b0:b0 + SMALL], part), b0
    assert np.array_equal(_batch(w, source, data, B), full)   # repeated: the scratch sets are reused
    w.close()


@pytest.mark.parametrize("kernel", [0, 1])
def test_submitted_chunked_batches_equal_synchronous_calls(bf, kernel):
    """Three chunked batches submitted back to back (a third submit waits for the oldest) deliver the bits of the
    synchronous calls, into the buffers they were submitted with."""
    import torch
    w = bf.MIMOWorker(cases.origins(1, 1), 16, 16, 180.0)
    w.set_kernel(kernel)
    base = _stream(B)
    T = base.shape[1]
    streams = [torch.from_numpy(base * np.float32(1.0 + 0.25 * k)).pin_memory() for k in range(3)]
    want = [w.power_map_batch(s.numpy(), B) for s in streams]
    outs = [torch.zeros((B, 256), dtype=torch.float32).pin_memory() for _ in range(3)]
    for k in range(3):
        w.power_map_batch_submit_ptr(streams[k].data_ptr(), T, B, outs[k].data_ptr())
    for _ in range(2):
        w.power_map_batch_wait()
    for k in range(3):
        assert np.array_equal(outs[k].numpy(), want[k]), k
    w.close()
