"""The C-ABI shared library loads and exports every symbol include/bflk.h declares (no GPU needed),
and fails loudly -- no CPU fallback -- when no B200 is present."""
import ctypes
import os
import re
import shutil
import subprocess
import sys

import pytest

import bflk
from conftest import ROOT


def header_symbols():
    text = open(os.path.join(ROOT, "include", "bflk.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(bflk_[a-z0-9_]+)\s*\(", text)))


def test_header_and_binding_agree():
    assert header_symbols() == sorted(bflk.SYMBOLS)


def test_library_exports_every_symbol():
    assert os.path.exists(bflk.LIB_PATH), "libbflk.so not built: run beamforming-lk_b200/build.sh"
    L = bflk.load_library()
    for name in header_symbols():
        assert hasattr(L, name), name
    exported = subprocess.run(["nm", "-D", "--defined-only", bflk.LIB_PATH], capture_output=True, text=True).stdout
    for name in header_symbols():
        assert re.search(rf"\bT {name}\b", exported), name
    assert L.bflk_version() == 1


def test_library_is_built_for_sm_100a():
    # the toolkit's bin/ need not be on PATH: else take cuobjdump from beside the nvcc build.sh uses ($NVCC, by default
    # /usr/local/cuda/bin/nvcc)
    nvcc = os.environ.get("NVCC") or "/usr/local/cuda/bin/nvcc"
    cuobjdump = shutil.which("cuobjdump") or os.path.join(os.path.dirname(nvcc), "cuobjdump")
    out = subprocess.run([cuobjdump, "-lelf", bflk.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out, out


def test_default_config_matches_reference_constants():
    L = bflk.load_library()
    cfg = bflk.Config()
    L.bflk_default_config(ctypes.byref(cfg))
    # streams.hpp:28-32, antenna.h:16-20
    assert (cfg.n_channels, cfg.frame_len, cfg.history, cfg.window_len) == (64, 256, 256, 1024)
    assert cfg.sample_rate == 48828.0 and cfg.propagation_speed == 340.0


def test_create_rejects_bad_config():
    L = bflk.load_library()
    cfg = bflk.Config()
    L.bflk_default_config(ctypes.byref(cfg))
    cfg.window_len = 300            # cannot hold history + frame + 1
    h = ctypes.c_void_p()
    assert L.bflk_create(ctypes.byref(cfg), ctypes.byref(h)) == -1
    assert b"window_len" in L.bflk_last_error(None)
    assert not h.value


def test_no_cpu_fallback_without_gpu():
    """In a child process that sees no GPU (CUDA_VISIBLE_DEVICES empty), so that it runs where one is present too."""
    code = ("import sys; sys.path.insert(0, sys.argv[1]); import bflk\n"
            "try:\n    bflk.Beamformer()\nexcept bflk.BflkError as e:\n    print(e.code, e)\n")
    r = subprocess.run([sys.executable, "-c", code, os.path.dirname(os.path.dirname(bflk.__file__))],
                       env={**os.environ, "CUDA_VISIBLE_DEVICES": ""}, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert r.stdout.startswith("-4 ") and "no CPU fallback" in r.stdout, r.stdout


def test_launch_shape_of_small_calls():
    """bflk_launch_shape (pure arithmetic): the CTA shape of calls too small to fill a B200, as measured in
    profiles/r2c_latency_shapes.txt -- and the throughput shape (0) for everything that fills two waves of 16-warp CTAs."""
    import bflk
    # one live frame
    assert bflk.launch_shape(32, 32, 512) == (4, 1)                          # cfg3: 64 four-warp CTAs, one warp per scheduler
    assert bflk.launch_shape(32, 32, 512, channel_split=True) == (8, 4)      # 128 eight-warp CTAs in clusters of 4
    assert bflk.launch_shape(64, 64, 256) == (8, 1)                          # cfg2: 128 CTAs
    assert bflk.launch_shape(64, 64, 256, channel_split=True) == (16, 2)
    assert bflk.launch_shape(100, 100, 64) == (12, 1)                        # cfg1: 209 CTAs in two waves beat 157 in two
    assert bflk.launch_shape(100, 100, 64, channel_split=True) == (12, 1)    # 8 stages: nothing to split
    # batches that fill the GPU keep the throughput shape, with or without the option
    for split in (False, True):
        assert bflk.launch_shape(32, 32, 512, n_frames=592, channel_split=split) == (0, 1)
        assert bflk.launch_shape(256, 256, 512, n_frames=1, frame_len=4096, channel_split=split) == (0, 1)
    # every answer is launchable: 2..16 warps, cluster of 1 / 2 / 4, at least 4 pipeline stages per rank
    for rows, cols, ch, nf in [(2, 2, 64, 1), (8, 8, 64, 3), (9, 9, 512, 1), (24, 24, 256, 6), (32, 32, 512, 5), (16, 128, 448, 2)]:
        for split in (False, True):
            for sms in (148, 132, 8):
                w, s = bflk.launch_shape(rows, cols, ch, n_frames=nf, n_sms=sms, channel_split=split)
                assert (w == 0 or 2 <= w <= 16) and s in (1, 2, 4) and (split or s == 1)
                assert s == 1 or ((ch + 7) // 8) // s >= 4
    with pytest.raises(bflk.BflkError):
        bflk.launch_shape(0, 32, 512)
