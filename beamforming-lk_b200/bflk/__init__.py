"""bflk -- Python host binding (ctypes) of the B200-native delay-and-sum library.

The product is ``libbflk.so`` (CUDA kernels for sm_100a behind the C ABI in ``include/bflk.h``); this
module only marshals numpy / torch buffers into that ABI.  There is no CPU fallback: if the shared
library is missing or no B200 is visible, construction raises.

Class names mirror the reference's workers (src/dsp/mimo.h, src/dsp/miso.h): ``MIMOWorker`` produces
the full-grid power map, ``MISOWorker`` the dynamically steered audio + beam power.
"""
import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.path.join(_PKG, "libbflk.so")

N_SAMPLES = 256       # src/fpga/streams.hpp:28
WINDOW = 1024         # N_ITEMS_BUFFER, src/fpga/streams.hpp:30-32
ELEMENTS = 64         # src/geometry/antenna.h:20
SAMPLE_RATE = 48828.0
PROPAGATION_SPEED = 340.0

KERNEL_AUTO, KERNEL_GENERIC, KERNEL_TILED, KERNEL_BCAST, KERNEL_TILED_FMA2 = 0, 1, 2, 3, 4

# every symbol include/bflk.h declares (tests check the library exports exactly these)
SYMBOLS = [
    "bflk_default_config", "bflk_version", "bflk_create", "bflk_destroy", "bflk_last_error",
    "bflk_set_geometry", "bflk_set_tiled_geometry", "bflk_get_geometry", "bflk_set_channel_mask",
    "bflk_set_grid_fov", "bflk_set_grid_tables", "bflk_set_grid_shape", "bflk_set_direction_range", "bflk_get_n_directions",
    "bflk_get_grid", "bflk_get_tables", "bflk_steer_tables", "bflk_power_map", "bflk_power_map_i32",
    "bflk_power_map_batch", "bflk_power_map_batch_submit", "bflk_power_map_batch_wait", "bflk_power_map_batch_i32", "bflk_power_map_batch_i32_dev",
    "bflk_power_map_batch_dev", "bflk_beams_batch_dev", "bflk_power_map_batch_dev_submit", "bflk_power_map_batch_dev_join", "bflk_set_kernel", "bflk_set_channel_split", "bflk_launch_shape", "bflk_get_kernel", "bflk_launch_count", "bflk_enable_timing",
    "bflk_kernel_time_ms", "bflk_fp32_peak_tflops", "bflk_set_window", "bflk_set_window_dev", "bflk_miso", "bflk_miso_dev", "bflk_monopulse", "bflk_set_fir",
    "bflk_pin_host", "bflk_unpin_host", "bflk_heatmap", "bflk_resize_u8", "bflk_targets", "bflk_targets_batch_dev", "bflk_calibrate", "bflk_ingest_i32",
    "bflk_stream_open", "bflk_stream_close", "bflk_stream_push", "bflk_stream_push_i32", "bflk_stream_power_maps",
    "bflk_stream_discard", "bflk_stream_status", "bflk_stream_window", "bflk_session_beams", "bflk_session_targets",
    "bflk_comm_unique_id", "bflk_comm_init_rank", "bflk_comm_info", "bflk_shard_plan",
    "bflk_power_map_batch_sharded_dev", "bflk_power_map_batch_sharded_dev_submit", "bflk_power_map_batch_sharded_dev_join", "bflk_power_map_batch_sharded", "bflk_power_map_batch_sharded_submit", "bflk_power_map_batch_sharded_wait",
    "bflk_group_create", "bflk_group_destroy", "bflk_group_size", "bflk_group_handle", "bflk_group_last_error",
    "bflk_group_set_geometry", "bflk_group_set_tiled_geometry", "bflk_group_set_channel_mask", "bflk_group_set_grid_fov",
    "bflk_group_set_kernel", "bflk_group_power_map_batch", "bflk_group_power_map_batch_dev", "bflk_group_synchronize",
]


class Config(C.Structure):
    _fields_ = [("n_channels", C.c_int32), ("frame_len", C.c_int32), ("history", C.c_int32),
                ("window_len", C.c_int32), ("sample_rate", C.c_double), ("propagation_speed", C.c_double),
                ("device", C.c_int32), ("reserved", C.c_int32)]


class Target(C.Structure):
    """struct bflk_target (Target of src/dsp/worker.h:32-61 for a peak of the MIMO map)."""
    _fields_ = [("theta", C.c_double), ("phi", C.c_double), ("power", C.c_float), ("probability", C.c_float),
                ("direction", C.c_int32), ("row", C.c_int32), ("col", C.c_int32), ("reserved", C.c_int32)]


# the same 40-byte record as a numpy dtype: decodes targets copied back from a device buffer (Beamformer.targets_batch_dev)
TARGET_DTYPE = np.dtype([("theta", np.float64), ("phi", np.float64), ("power", np.float32), ("probability", np.float32),
                         ("direction", np.int32), ("row", np.int32), ("col", np.int32), ("reserved", np.int32)])
assert TARGET_DTYPE.itemsize == C.sizeof(Target)


def decode_targets(raw, counts):
    """Records of a [n_maps][max_targets] buffer of bflk_target (raw bytes or a uint8 / TARGET_DTYPE array of that size) and
    counts [n_maps] -> one list of target dicts per map, as Beamformer.targets returns them."""
    counts = np.asarray(counts).ravel()
    rec = np.frombuffer(np.ascontiguousarray(raw).tobytes() if not isinstance(raw, bytes) else raw, TARGET_DTYPE)
    rec = rec.reshape(counts.shape[0], -1)
    keys = ("theta", "phi", "power", "probability", "direction", "row", "col")
    return [[{k: t[k].item() for k in keys} for t in rec[b, :counts[b]]] for b in range(counts.shape[0])]


class BflkError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"bflk error {code}: {msg}")
        self.code = code


_lib = None


def load_library():
    """Load libbflk.so (fails loudly when the CUDA extension has not been built)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with beamforming-lk_b200/build.sh "
                          "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, f32, f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_double
    L.bflk_default_config.argtypes = [C.POINTER(Config)]
    L.bflk_default_config.restype = None
    L.bflk_version.restype = C.c_int
    L.bflk_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    L.bflk_destroy.argtypes = [vp]
    L.bflk_last_error.argtypes = [vp]
    L.bflk_last_error.restype = C.c_char_p
    L.bflk_set_geometry.argtypes = [vp, vp, i32]
    L.bflk_set_tiled_geometry.argtypes = [vp, i32, vp]
    L.bflk_get_geometry.argtypes = [vp, vp]
    L.bflk_set_channel_mask.argtypes = [vp, vp, i32]
    L.bflk_set_grid_fov.argtypes = [vp, i32, i32, f32]
    L.bflk_set_grid_tables.argtypes = [vp, vp, vp, i32]
    L.bflk_set_grid_shape.argtypes = [vp, i32, i32]
    L.bflk_set_direction_range.argtypes = [vp, i32, i32]
    L.bflk_get_n_directions.argtypes = [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]
    L.bflk_get_grid.argtypes = [vp, vp, vp]
    L.bflk_get_tables.argtypes = [vp, vp, vp]
    L.bflk_steer_tables.argtypes = [vp, vp, vp, i32, vp, vp]
    L.bflk_power_map.argtypes = [vp, vp, vp]
    L.bflk_power_map_i32.argtypes = [vp, vp, vp]
    L.bflk_power_map_batch.argtypes = [vp, vp, i64, i32, vp]
    L.bflk_power_map_batch_submit.argtypes = [vp, vp, i64, i32, vp]
    L.bflk_power_map_batch_wait.argtypes = [vp]
    L.bflk_power_map_batch_i32.argtypes = [vp, vp, i64, i32, vp]
    L.bflk_power_map_batch_i32_dev.argtypes = [vp, vp, i64, i32, vp, vp]
    L.bflk_power_map_batch_dev.argtypes = [vp, vp, i64, i32, vp, vp]
    L.bflk_beams_batch_dev.argtypes = [vp, vp, i64, i32, vp, vp, vp]
    L.bflk_power_map_batch_dev_submit.argtypes = [vp, vp, i64, i32, vp, vp]
    L.bflk_power_map_batch_dev_join.argtypes = [vp, vp]
    L.bflk_set_kernel.argtypes = [vp, i32]
    L.bflk_set_channel_split.argtypes = [vp, i32]
    L.bflk_launch_shape.argtypes = [i32, i32, i32, i32, i32, i32, i32, C.POINTER(i32), C.POINTER(i32)]
    L.bflk_launch_count.argtypes = [vp]
    L.bflk_launch_count.restype = i64
    L.bflk_get_kernel.argtypes = [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]
    L.bflk_enable_timing.argtypes = [vp, i32]
    L.bflk_kernel_time_ms.argtypes = [vp, C.POINTER(f32), C.POINTER(i32), C.POINTER(f32), C.POINTER(i32)]
    L.bflk_fp32_peak_tflops.argtypes = [vp, C.POINTER(f32)]
    L.bflk_set_window.argtypes = [vp, vp]
    L.bflk_set_window_dev.argtypes = [vp, vp]
    L.bflk_miso.argtypes = [vp, vp, vp, i32, vp, vp, vp]
    L.bflk_miso_dev.argtypes = [vp, vp, vp, i32, vp, vp, vp, vp]
    L.bflk_monopulse.argtypes = [vp, vp, vp, i32, C.c_double, C.c_double, C.c_double, vp, vp, vp, vp, vp, vp]
    L.bflk_set_fir.argtypes = [vp, vp, i32, i32]
    L.bflk_heatmap.argtypes = [vp, vp, i32, vp, C.POINTER(i32), C.POINTER(f32)]
    L.bflk_pin_host.argtypes = [vp, C.c_size_t]
    L.bflk_unpin_host.argtypes = [vp]
    L.bflk_resize_u8.argtypes = [vp, vp, i32, i32, i32, i32, vp]
    L.bflk_targets.argtypes = [vp, vp, i32, f32, vp, C.POINTER(i32)]
    L.bflk_targets_batch_dev.argtypes = [vp, vp, i32, i32, f32, vp, vp, vp]
    L.bflk_calibrate.argtypes = [vp, vp, i32, f32, vp, vp, C.POINTER(i32), C.POINTER(f32), C.POINTER(f32)]
    L.bflk_ingest_i32.argtypes = [vp, vp, i32, i32, vp]
    L.bflk_stream_open.argtypes = [vp, i32]
    L.bflk_stream_close.argtypes = [vp]
    L.bflk_stream_push.argtypes = [vp, vp, i32]
    L.bflk_stream_push_i32.argtypes = [vp, vp, i32]
    L.bflk_stream_power_maps.argtypes = [vp, i32, vp, C.POINTER(i64), C.POINTER(i32)]
    L.bflk_session_beams.argtypes = [vp, i32, vp, vp, C.POINTER(i64), C.POINTER(i32)]
    L.bflk_session_targets.argtypes = [vp, i32, i32, f32, vp, vp, vp, C.POINTER(i64), C.POINTER(i32)]
    L.bflk_stream_discard.argtypes = [vp, i32]
    L.bflk_stream_status.argtypes = [vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(i32), C.POINTER(i64)]
    L.bflk_stream_window.argtypes = [vp, i64]
    L.bflk_comm_unique_id.argtypes = [vp]
    L.bflk_comm_init_rank.argtypes = [vp, vp, i32, i32, i32]
    L.bflk_comm_info.argtypes = [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i64)]
    L.bflk_shard_plan.argtypes = [i32, i32, i32, i32, i32, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]
    L.bflk_power_map_batch_sharded_dev.argtypes = [vp, vp, i64, i32, vp, vp]
    L.bflk_power_map_batch_sharded_dev_submit.argtypes = [vp, vp, i64, i32, vp, vp]
    L.bflk_power_map_batch_sharded_dev_join.argtypes = [vp, vp]
    L.bflk_power_map_batch_sharded.argtypes = [vp, vp, i64, i32, vp]
    L.bflk_power_map_batch_sharded_submit.argtypes = [vp, vp, i64, i32, vp]
    L.bflk_power_map_batch_sharded_wait.argtypes = [vp]
    L.bflk_group_create.argtypes = [C.POINTER(Config), vp, i32, i32, C.POINTER(vp)]
    L.bflk_group_destroy.argtypes = [vp]
    L.bflk_group_size.argtypes = [vp]
    L.bflk_group_size.restype = i32
    L.bflk_group_handle.argtypes = [vp, i32]
    L.bflk_group_handle.restype = vp
    L.bflk_group_last_error.argtypes = [vp]
    L.bflk_group_last_error.restype = C.c_char_p
    L.bflk_group_set_geometry.argtypes = [vp, vp, i32]
    L.bflk_group_set_tiled_geometry.argtypes = [vp, i32, vp]
    L.bflk_group_set_channel_mask.argtypes = [vp, vp, i32]
    L.bflk_group_set_grid_fov.argtypes = [vp, i32, i32, f32]
    L.bflk_group_set_kernel.argtypes = [vp, i32]
    L.bflk_group_power_map_batch.argtypes = [vp, vp, i64, i32, vp]
    L.bflk_group_power_map_batch_dev.argtypes = [vp, vp, i64, i32, vp]
    L.bflk_group_synchronize.argtypes = [vp]
    _lib = L
    return L


def _np(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def shard_plan(n_directions, n_frames, n_ranks, rank, dir_groups=0):
    """(dir_first, dir_count, frame_first, frame_count) of rank `rank` (bflk_shard_plan; needs no device)."""
    L = load_library()
    a, b, c, d = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
    rc = L.bflk_shard_plan(n_directions, n_frames, n_ranks, dir_groups, rank, C.byref(a), C.byref(b), C.byref(c), C.byref(d))
    if rc != 0:
        raise BflkError(rc, f"bflk_shard_plan({n_directions}, {n_frames}, {n_ranks}, {dir_groups}, {rank})")
    return a.value, b.value, c.value, d.value


def launch_shape(rows, cols, n_channels, n_frames=1, frame_len=256, n_sms=148, channel_split=False):
    """(warps per CTA, cluster size of the channel split) a power-map call gets (bflk_launch_shape; needs no device)."""
    L = load_library()
    w, s = C.c_int32(), C.c_int32()
    rc = L.bflk_launch_shape(rows, cols, n_channels, frame_len, n_frames, n_sms, 1 if channel_split else 0, C.byref(w), C.byref(s))
    if rc != 0:
        raise BflkError(rc, f"bflk_launch_shape({rows}, {cols}, {n_channels}, {frame_len}, {n_frames}, {n_sms})")
    return w.value, s.value


def comm_unique_id():
    """128 bytes identifying a new multi-GPU job (rank 0 creates it, the caller broadcasts it)."""
    L = load_library()
    buf = (C.c_uint8 * 128)()
    rc = L.bflk_comm_unique_id(buf)
    if rc != 0:
        raise BflkError(rc, "bflk_comm_unique_id: NCCL is not available")
    return bytes(buf)


def tile_origins(nx, ny, pitch=0.16):
    """Origins of nx x ny abutting 8x8 arrays (0.16 m pitch), centred, row-major: tile a = j*nx + i."""
    o = [[(i - (nx - 1) / 2) * pitch, (j - (ny - 1) / 2) * pitch, 0.0] for j in range(ny) for i in range(nx)]
    return np.asarray(o, np.float32)


class Beamformer:
    """Thin object wrapper over a ``bflk_handle``."""

    def __init__(self, n_channels=ELEMENTS, frame_len=N_SAMPLES, history=N_SAMPLES, window_len=WINDOW,
                 sample_rate=SAMPLE_RATE, propagation_speed=PROPAGATION_SPEED, device=0):
        self._L = load_library()
        cfg = Config()
        self._L.bflk_default_config(C.byref(cfg))
        cfg.n_channels, cfg.frame_len, cfg.history, cfg.window_len = n_channels, frame_len, history, window_len
        cfg.sample_rate, cfg.propagation_speed, cfg.device = sample_rate, propagation_speed, device
        self.cfg = cfg
        self._h = C.c_void_p()
        rc = self._L.bflk_create(C.byref(cfg), C.byref(self._h))
        if rc != 0:
            raise BflkError(rc, self._L.bflk_last_error(None).decode())

    # -- plumbing -----------------------------------------------------------------------------------------
    def _check(self, rc):
        if rc != 0:
            raise BflkError(rc, self._L.bflk_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._L.bflk_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def n_channels(self):
        return self.cfg.n_channels

    @property
    def frame_len(self):
        return self.cfg.frame_len

    def launch_count(self):
        return int(self._L.bflk_launch_count(self._h))

    # -- multi-GPU: this handle as one rank of a job (one process per GPU) ---------------------------------------
    def comm_init_rank(self, unique_id, n_ranks, rank, dir_groups=0):
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        self._check(self._L.bflk_comm_init_rank(self._h, buf, n_ranks, rank, dir_groups))

    def comm_info(self):
        """(n_ranks, rank, direction groups, frame groups, collectives issued so far)."""
        a, b, c, d, e = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32(), C.c_int64()
        self._check(self._L.bflk_comm_info(self._h, C.byref(a), C.byref(b), C.byref(c), C.byref(d), C.byref(e)))
        return a.value, b.value, c.value, d.value, e.value

    def power_map_batch_sharded_dev(self, stream_dev_ptr, n_samples, n_frames, power_all_dev_ptr, cuda_stream=0):
        self._check(self._L.bflk_power_map_batch_sharded_dev(self._h, C.c_void_p(stream_dev_ptr), n_samples, n_frames,
                                                             C.c_void_p(power_all_dev_ptr), C.c_void_p(cuda_stream)))

    def power_map_batch_sharded_dev_submit(self, stream_dev_ptr, n_samples, n_frames, power_all_dev_ptr, cuda_stream=0):
        """kernels on cuda_stream, all-gather + assembly on the communicator's stream (bflk.h); complete after _dev_join"""
        self._check(self._L.bflk_power_map_batch_sharded_dev_submit(self._h, C.c_void_p(stream_dev_ptr), n_samples, n_frames,
                                                                    C.c_void_p(power_all_dev_ptr), C.c_void_p(cuda_stream)))

    def power_map_batch_sharded_dev_join(self, cuda_stream=0):
        self._check(self._L.bflk_power_map_batch_sharded_dev_join(self._h, C.c_void_p(cuda_stream)))

    def power_map_batch_sharded_submit_ptr(self, stream_ptr, n_samples, n_frames, power_ptr):
        self._check(self._L.bflk_power_map_batch_sharded_submit(self._h, C.c_void_p(stream_ptr), n_samples, n_frames,
                                                                C.c_void_p(power_ptr) if power_ptr else None))

    def power_map_batch_sharded_wait(self):
        self._check(self._L.bflk_power_map_batch_sharded_wait(self._h))

    def power_map_batch_sharded_ptr(self, stream_ptr, n_samples, n_frames, power_ptr):
        self._check(self._L.bflk_power_map_batch_sharded(self._h, C.c_void_p(stream_ptr), n_samples, n_frames,
                                                         C.c_void_p(power_ptr) if power_ptr else None))

    def kernel_info(self):
        """(last kernel used: 1 generic / 2 tiled exact / 3 lane-broadcast / 4 tiled two-FMA / 0 none yet, largest offset
        spread of a direction tile in the mode the grid tiles with (-1 before the tiles are built), window chunks of the
        tiled variant (0 when the grid does not tile))."""
        a, b, c = C.c_int32(), C.c_int32(), C.c_int32()
        self._check(self._L.bflk_get_kernel(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def fp32_peak_tflops(self):
        """TFLOP/s of a packed-FMA saturation kernel on this device (empirical FP32 roofline)."""
        v = C.c_float()
        self._check(self._L.bflk_fp32_peak_tflops(self._h, C.byref(v)))
        return v.value

    def enable_timing(self, on=True):
        self._check(self._L.bflk_enable_timing(self._h, 1 if on else 0))

    def kernel_time_ms(self):
        """(das_ms, das_launches, pack_ms, pack_launches) accumulated since the last call."""
        a, b, c, d = C.c_float(), C.c_int32(), C.c_float(), C.c_int32()
        self._check(self._L.bflk_kernel_time_ms(self._h, C.byref(a), C.byref(b), C.byref(c), C.byref(d)))
        return a.value, b.value, c.value, d.value

    # -- geometry / tables ------------------------------------------------------------------------------------
    def set_geometry(self, xyz):
        xyz = _np(xyz, np.float32).reshape(-1, 3)
        self._check(self._L.bflk_set_geometry(self._h, _ptr(xyz), xyz.shape[0]))

    def set_tiled_geometry(self, origins):
        origins = _np(origins, np.float32).reshape(-1, 3)
        self._check(self._L.bflk_set_tiled_geometry(self._h, origins.shape[0], _ptr(origins)))

    def geometry(self):
        xyz = np.zeros((self.n_channels, 3), np.float32)
        self._check(self._L.bflk_get_geometry(self._h, _ptr(xyz)))
        return xyz

    def set_channel_mask(self, index=None):
        if index is None:
            self._check(self._L.bflk_set_channel_mask(self._h, None, 0))
        else:
            index = _np(index, np.int32)
            self._check(self._L.bflk_set_channel_mask(self._h, _ptr(index), index.shape[0]))

    def set_grid_fov(self, rows, cols, fov_deg):
        self._check(self._L.bflk_set_grid_fov(self._h, rows, cols, float(fov_deg)))

    def set_grid_tables(self, offsets, fractions):
        offsets, fractions = _np(offsets, np.int32), _np(fractions, np.float32)
        assert offsets.shape == fractions.shape and offsets.shape[1] == self.n_channels
        self._check(self._L.bflk_set_grid_tables(self._h, _ptr(offsets), _ptr(fractions), offsets.shape[0]))

    def set_grid_shape(self, rows, cols):
        """Caller-supplied tables are a row-major rows x cols grid: lets the register-tiled kernels serve them."""
        self._check(self._L.bflk_set_grid_shape(self._h, rows, cols))

    def set_direction_range(self, first, count):
        self._check(self._L.bflk_set_direction_range(self._h, first, count))

    def n_directions(self):
        t, f, c = C.c_int32(), C.c_int32(), C.c_int32()
        self._check(self._L.bflk_get_n_directions(self._h, C.byref(t), C.byref(f), C.byref(c)))
        return t.value, f.value, c.value

    def grid(self):
        D = self.n_directions()[0]
        th, ph = np.zeros(D, np.float64), np.zeros(D, np.float64)
        self._check(self._L.bflk_get_grid(self._h, _ptr(th), _ptr(ph)))
        return th, ph

    def tables(self):
        D = self.n_directions()[0]
        off = np.zeros((D, self.n_channels), np.int32)
        fr = np.zeros((D, self.n_channels), np.float32)
        self._check(self._L.bflk_get_tables(self._h, _ptr(off), _ptr(fr)))
        return off, fr

    def steer_tables(self, theta, phi):
        theta, phi = _np(theta, np.float64).ravel(), _np(phi, np.float64).ravel()
        T = theta.shape[0]
        off = np.zeros((T, self.n_channels), np.int32)
        fr = np.zeros((T, self.n_channels), np.float32)
        self._check(self._L.bflk_steer_tables(self._h, _ptr(theta), _ptr(phi), T, _ptr(off), _ptr(fr)))
        return off, fr

    def set_kernel(self, which):
        self._check(self._L.bflk_set_kernel(self._h, which))

    def set_channel_split(self, on):
        """latency option of small two-FMA calls: channels split across a thread-block cluster (bflk.h)"""
        self._check(self._L.bflk_set_channel_split(self._h, 1 if on else 0))

    # -- hot path -----------------------------------------------------------------------------------------------
    def power_map(self, window):
        """window [C][W] float32 (host) -> power [count] (MIMOWorker::update)."""
        window = _np(window, np.float32)
        assert window.shape == (self.n_channels, self.cfg.window_len), window.shape
        out = np.zeros(self.n_directions()[2], np.float32)
        self._check(self._L.bflk_power_map(self._h, _ptr(window), _ptr(out)))
        return out

    def power_map_i32(self, frames):
        """frames [W][C] int32 wire samples (one row per time sample) -> power [count]."""
        frames = _np(frames, np.int32)
        assert frames.shape == (self.cfg.window_len, self.n_channels), frames.shape
        out = np.zeros(self.n_directions()[2], np.float32)
        self._check(self._L.bflk_power_map_i32(self._h, _ptr(frames), _ptr(out)))
        return out

    def power_map_batch_i32(self, frames, n_frames):
        """frames [T][C] int32 wire samples (one row per time sample), frame b at row b*N -> power [B][count]."""
        frames = _np(frames, np.int32)
        assert frames.shape[1] == self.n_channels
        out = np.zeros((n_frames, self.n_directions()[2]), np.float32)
        self._check(self._L.bflk_power_map_batch_i32(self._h, _ptr(frames), frames.shape[0], n_frames, _ptr(out)))
        return out

    def power_map_batch_i32_dev(self, frames_dev_ptr, n_samples, n_frames, power_dev_ptr, cuda_stream=0):
        """Device wire rows [T][C] int32 (e.g. a torch tensor's data_ptr()) -> power [B][count] on the device, asynchronous."""
        self._check(self._L.bflk_power_map_batch_i32_dev(self._h, C.c_void_p(frames_dev_ptr), n_samples, n_frames,
                                                         C.c_void_p(power_dev_ptr), C.c_void_p(cuda_stream)))

    def power_map_batch(self, stream, n_frames):
        """stream [C][T] float32 (host), frame b at sample b*N -> power [B][count]."""
        stream = _np(stream, np.float32)
        assert stream.shape[0] == self.n_channels
        out = np.zeros((n_frames, self.n_directions()[2]), np.float32)
        self._check(self._L.bflk_power_map_batch(self._h, _ptr(stream), stream.shape[1], n_frames, _ptr(out)))
        return out

    def power_map_batch_ptr(self, stream_ptr, n_samples, n_frames, power_ptr, cuda_stream=0):
        """Raw host-pointer variant (pinned buffers) -- what bench.py's e2e leg calls."""
        self._check(self._L.bflk_power_map_batch(self._h, C.c_void_p(stream_ptr), n_samples, n_frames, C.c_void_p(power_ptr)))

    def power_map_batch_submit_ptr(self, stream_ptr, n_samples, n_frames, power_ptr):
        """Asynchronous host batch (page-locked buffers): enqueue and return; at most two batches in flight."""
        self._check(self._L.bflk_power_map_batch_submit(self._h, C.c_void_p(stream_ptr), n_samples, n_frames, C.c_void_p(power_ptr)))

    def power_map_batch_wait(self):
        """Blocks until the oldest submitted batch has delivered its maps."""
        self._check(self._L.bflk_power_map_batch_wait(self._h))

    def power_map_batch_dev(self, stream_dev_ptr, n_samples, n_frames, power_dev_ptr, cuda_stream=0):
        """Device pointers (e.g. torch tensors' data_ptr()), asynchronous on cuda_stream."""
        self._check(self._L.bflk_power_map_batch_dev(self._h, C.c_void_p(stream_dev_ptr), n_samples, n_frames,
                                                     C.c_void_p(power_dev_ptr), C.c_void_p(cuda_stream)))

    def beams_batch_dev(self, stream_dev_ptr, n_samples, n_frames, beams_dev_ptr, power_dev_ptr, cuda_stream=0):
        """power_map_batch_dev that also writes the delayed sums its maps square: beams [B][count][N] (device, 8-byte aligned)."""
        self._check(self._L.bflk_beams_batch_dev(self._h, C.c_void_p(stream_dev_ptr), n_samples, n_frames,
                                                 C.c_void_p(beams_dev_ptr), C.c_void_p(power_dev_ptr), C.c_void_p(cuda_stream)))

    def power_map_batch_dev_submit(self, stream_dev_ptr, n_samples, n_frames, power_dev_ptr, cuda_stream=0):
        """Continuous operation (bflk.h): consecutive batches overlap on the handle's two compute streams; complete after _dev_join."""
        self._check(self._L.bflk_power_map_batch_dev_submit(self._h, C.c_void_p(stream_dev_ptr), n_samples, n_frames,
                                                            C.c_void_p(power_dev_ptr), C.c_void_p(cuda_stream)))

    def power_map_batch_dev_join(self, cuda_stream=0):
        self._check(self._L.bflk_power_map_batch_dev_join(self._h, C.c_void_p(cuda_stream)))

    def set_window(self, window):
        """Keep window [C][W] on the device: miso() / monopulse() with window=None then work on it (None forgets it)."""
        if window is None:
            self._check(self._L.bflk_set_window(self._h, None))
            return
        window = _np(window, np.float32)
        assert window.shape == (self.n_channels, self.cfg.window_len), window.shape
        self._check(self._L.bflk_set_window(self._h, _ptr(window)))

    def miso(self, theta, phi, window=None, want_audio=True, want_power=True):
        """Particle::steer + das + beam for T targets: returns (audio [T][N] | None, power [T] | None).
        window=None: the window kept on the device by set_window()."""
        theta, phi = _np(theta, np.float64).ravel(), _np(phi, np.float64).ravel()
        if window is not None:
            window = _np(window, np.float32)
            assert window.shape == (self.n_channels, self.cfg.window_len), window.shape
        T = theta.shape[0]
        audio = np.zeros((T, self.frame_len), np.float32) if want_audio else None
        power = np.zeros(T, np.float32) if want_power else None
        self._check(self._L.bflk_miso(self._h, _ptr(theta), _ptr(phi), T, _ptr(window) if window is not None else None,
                                      _ptr(audio) if want_audio else None, _ptr(power) if want_power else None))
        return audio, power

    def set_window_dev(self, window_dev_ptr):
        """Borrow a device window [C][W] float32 (e.g. a torch tensor's data_ptr()) as the resident one; 0 / None forgets it.
        The buffer must outlive its use: the handle does not copy it."""
        self._check(self._L.bflk_set_window_dev(self._h, C.c_void_p(window_dev_ptr) if window_dev_ptr else None))

    def miso_dev(self, theta, phi, window_dev_ptr, audio_dev_ptr, power_dev_ptr, cuda_stream=0):
        """miso() on device buffers, asynchronous on cuda_stream: window [C][W] (None: the resident window), audio [T][N]
        and power [T] (either may be 0 / None).  A delay beyond the history is clamped to it, not reported (bflk.h)."""
        theta, phi = _np(theta, np.float64).ravel(), _np(phi, np.float64).ravel()
        ptr = lambda p: C.c_void_p(p) if p else None
        self._check(self._L.bflk_miso_dev(self._h, _ptr(theta), _ptr(phi), theta.shape[0], ptr(window_dev_ptr),
                                          ptr(audio_dev_ptr), ptr(power_dev_ptr), C.c_void_p(cuda_stream)))

    def set_fir(self, coeffs):
        """FIR interpolation of the reference's USE_FILTER build (delay.cpp:28-40): coeffs [n_phases][taps], None = 2-tap form."""
        if coeffs is None:
            self._check(self._L.bflk_set_fir(self._h, None, 0, 0))
            return
        coeffs = _np(coeffs, np.float32)
        self._check(self._L.bflk_set_fir(self._h, _ptr(coeffs), coeffs.shape[0], coeffs.shape[1]))

    def monopulse(self, theta, phi, window, spread, theta_limit, reference=0.0):  # window=None: the resident window
        """GradientParticle::findNearby + the beam part of step() for P particles: returns (theta' [P], near_theta [P][4],
        near_phi [P][4], q [P][4], gradient [P][3] = (theta, phi, radius), error [P])."""
        theta, phi = _np(theta, np.float64).ravel().copy(), _np(phi, np.float64).ravel()
        if window is not None:
            window = _np(window, np.float32)
            assert window.shape == (self.n_channels, self.cfg.window_len), window.shape
        P = theta.shape[0]
        nth, nph, q = np.zeros((P, 4)), np.zeros((P, 4)), np.zeros((P, 4))
        grad, err = np.zeros((P, 3)), np.zeros(P)
        self._check(self._L.bflk_monopulse(self._h, _ptr(theta), _ptr(phi), P, C.c_double(spread), C.c_double(theta_limit),
                                           C.c_double(reference), _ptr(window) if window is not None else None, _ptr(nth), _ptr(nph), _ptr(q), _ptr(grad), _ptr(err)))
        return theta, nth, nph, q, grad, err

    # -- streaming session (bflk.h: bflk_stream_*) ----------------------------------------------------------------
    def stream_open(self, max_frames):
        """(Re)start a session at sample 0 with device history for max_frames ready frames."""
        self._check(self._L.bflk_stream_open(self._h, max_frames))

    def stream_close(self):
        self._check(self._L.bflk_stream_close(self._h))

    def stream_push(self, samples):
        """samples [C][n] float32, the next n samples of every channel."""
        samples = _np(samples, np.float32)
        assert samples.ndim == 2 and samples.shape[0] == self.n_channels, samples.shape
        self._check(self._L.bflk_stream_push(self._h, _ptr(samples), samples.shape[1]))

    def stream_push_i32(self, rows):
        """rows [n][C] int32 wire samples, one row per time sample."""
        rows = _np(rows, np.int32)
        assert rows.ndim == 2 and rows.shape[1] == self.n_channels, rows.shape
        self._check(self._L.bflk_stream_push_i32(self._h, _ptr(rows), rows.shape[0]))

    def stream_power_maps(self, max_frames=1):
        """Maps the oldest ready frames (at most max_frames) in one call: (first_frame, power [n][count]), n may be 0."""
        out = np.zeros((max_frames, self.n_directions()[2]), np.float32)
        first, n = C.c_int64(), C.c_int32()
        self._check(self._L.bflk_stream_power_maps(self._h, max_frames, _ptr(out), C.byref(first), C.byref(n)))
        return first.value, out[:n.value].copy()

    def stream_beams(self, max_frames=1):
        """stream_power_maps with the frames' beams: (first_frame, beams [n][count][N], power [n][count]), n may be 0."""
        count = self.n_directions()[2]
        beams = np.zeros((max_frames, count, self.frame_len), np.float32)
        out = np.zeros((max_frames, count), np.float32)
        first, n = C.c_int64(), C.c_int32()
        self._check(self._L.bflk_session_beams(self._h, max_frames, _ptr(beams), _ptr(out), C.byref(first), C.byref(n)))
        return first.value, beams[:n.value].copy(), out[:n.value].copy()

    def stream_targets(self, max_frames=1, max_targets=8, min_rel_power=0.5):
        """stream_power_maps with the Targets of every map: (first_frame, power [n][count], [list of target dicts per frame]),
        n may be 0."""
        count = self.n_directions()[2]
        out = np.zeros((max_frames, count), np.float32)
        recs = (Target * (max_frames * max_targets))()
        counts = np.zeros(max_frames, np.int32)
        first, n = C.c_int64(), C.c_int32()
        self._check(self._L.bflk_session_targets(self._h, max_frames, max_targets, float(min_rel_power), _ptr(out), recs,
                                                 _ptr(counts), C.byref(first), C.byref(n)))
        return first.value, out[:n.value].copy(), decode_targets(bytes(recs), counts)[:n.value]

    def stream_discard(self, keep=0):
        """Skip every ready frame but the newest `keep`."""
        self._check(self._L.bflk_stream_discard(self._h, keep))

    def stream_status(self):
        """(samples pushed per channel, next frame to map, frames ready, frames skipped)."""
        a, b, c, d = C.c_int64(), C.c_int64(), C.c_int32(), C.c_int64()
        self._check(self._L.bflk_stream_status(self._h, C.byref(a), C.byref(b), C.byref(c), C.byref(d)))
        return a.value, b.value, c.value, d.value

    def stream_window(self, frame):
        """Session frame `frame` becomes the resident window of miso() / monopulse() with window=None."""
        self._check(self._L.bflk_stream_window(self._h, frame))

    # -- neighbours ---------------------------------------------------------------------------------------------
    def heatmap(self, power):
        power = _np(power, np.float32).ravel()
        heat = np.zeros(power.shape[0], np.uint8)
        arg, mx = C.c_int32(), C.c_float()
        self._check(self._L.bflk_heatmap(self._h, _ptr(power), power.shape[0], _ptr(heat), C.byref(arg), C.byref(mx)))
        return heat, arg.value, mx.value

    def resize_u8(self, image, out_rows, out_cols):
        """cv::resize(image, (out_cols, out_rows), INTER_LINEAR) of an 8-bit map, bit-identical to OpenCV."""
        image = _np(image, np.uint8)
        out = np.zeros((out_rows, out_cols), np.uint8)
        self._check(self._L.bflk_resize_u8(self._h, _ptr(image), image.shape[0], image.shape[1], out_rows, out_cols, _ptr(out)))
        return out

    def targets(self, power=None, max_targets=8, min_rel_power=0.5):
        """Peaks of the map as Targets: list of dicts; power=None uses the map the last single-frame power_map left on the device."""
        arr = (Target * max_targets)()
        n = C.c_int32()
        if power is not None:
            power = _np(power, np.float32).ravel()
        self._check(self._L.bflk_targets(self._h, _ptr(power) if power is not None else None, max_targets, float(min_rel_power), arr, C.byref(n)))
        return [dict(theta=t.theta, phi=t.phi, power=t.power, probability=t.probability, direction=t.direction, row=t.row, col=t.col)
                for t in arr[:n.value]]

    def targets_batch_dev(self, power_dev_ptr, n_maps, targets_dev_ptr, n_dev_ptr, max_targets=8, min_rel_power=0.5,
                          cuda_stream=0):
        """Targets of n_maps whole-grid maps [n_maps][D] on the device, one launch, asynchronous on cuda_stream:
        targets_dev [n_maps][max_targets] bflk_target records (40 bytes each; decode_targets / TARGET_DTYPE read them back),
        n_dev [n_maps] int32 counts."""
        self._check(self._L.bflk_targets_batch_dev(self._h, C.c_void_p(power_dev_ptr), n_maps, max_targets, float(min_rel_power),
                                                   C.c_void_p(targets_dev_ptr), C.c_void_p(n_dev_ptr), C.c_void_p(cuda_stream)))

    def calibrate(self, signals, reference_power_level=1e-5):
        signals = _np(signals, np.float32)
        assert signals.shape[0] == ELEMENTS
        index = np.zeros(ELEMENTS, np.int32)
        corr = np.zeros(ELEMENTS, np.float32)
        n, med, mean = C.c_int32(), C.c_float(), C.c_float()
        self._check(self._L.bflk_calibrate(self._h, _ptr(signals), signals.shape[1], reference_power_level,
                                           _ptr(index), _ptr(corr), C.byref(n), C.byref(med), C.byref(mean)))
        return index[:n.value].copy(), corr[:n.value].copy(), med.value, mean.value

    def ingest_i32(self, frames):
        frames = _np(frames, np.int32)
        n, ns = frames.shape
        out = np.zeros((ns, n), np.float32)
        self._check(self._L.bflk_ingest_i32(self._h, _ptr(frames), n, ns, _ptr(out)))
        return out


class MIMOWorker(Beamformer):
    """Full-grid power map, constructor arguments as MIMOWorker(pipeline, antenna, running, rows, columns, fov)
    (src/dsp/mimo.h:36) with the antenna given as tile origins."""

    def __init__(self, origins, rows, columns, fov, index=None, device=0, **kw):
        origins = np.asarray(origins, np.float32).reshape(-1, 3)
        super().__init__(n_channels=ELEMENTS * origins.shape[0], device=device, **kw)
        self.set_tiled_geometry(origins)
        if index is not None:
            self.set_channel_mask(index)
        self.rows, self.columns, self.fov = rows, columns, fov
        self.set_grid_fov(rows, columns, fov)
        self.powerdB = np.zeros(rows * columns, np.float32)

    def update(self, window):
        """MIMOWorker::update (src/dsp/mimo.cpp:97-151) on a [C][W] snapshot."""
        self.powerdB = self.power_map(window)
        return self.powerdB

    def populateHeatmap(self):
        """MIMOWorker::populateHeatmap (src/dsp/mimo.cpp:61-95): uint8 [rows][columns]."""
        heat, arg, mx = self.heatmap(self.powerdB)
        return heat.reshape(self.rows, self.columns), arg, mx


class MISOWorker(Beamformer):
    """Dynamically steered DAS, MISOWorker(pipeline, antenna, running, fov) (src/dsp/miso.h:18), T targets."""

    def __init__(self, origins, fov=180.0, index=None, device=0, **kw):
        origins = np.asarray(origins, np.float32).reshape(-1, 3)
        super().__init__(n_channels=ELEMENTS * origins.shape[0], device=device, **kw)
        self.set_tiled_geometry(origins)
        if index is not None:
            self.set_channel_mask(index)
        self.fov = fov
        self.theta = np.zeros(1)
        self.phi = np.zeros(1)

    def steer(self, theta, phi):
        self.theta, self.phi = np.atleast_1d(theta).astype(np.float64), np.atleast_1d(phi).astype(np.float64)

    def update(self, window):
        """beamformer.steer(direction); beamformer.das(data) (src/dsp/miso.cpp:42-46) for every target."""
        return self.miso(self.theta, self.phi, window)


class Group:
    """One process, several GPUs (bflk_group_*): the grid (x the frames of a batch) sharded across `devices`."""

    def __init__(self, origins, rows, columns, fov, devices, dir_groups=0, frame_len=N_SAMPLES, history=N_SAMPLES,
                 window_len=WINDOW, kernel=0):
        self._L = load_library()
        origins = np.asarray(origins, np.float32).reshape(-1, 3)
        cfg = Config()
        self._L.bflk_default_config(C.byref(cfg))
        cfg.n_channels, cfg.frame_len, cfg.history, cfg.window_len = ELEMENTS * origins.shape[0], frame_len, history, window_len
        self.cfg = cfg
        devs = np.asarray(devices, np.int32)
        self._g = C.c_void_p()
        rc = self._L.bflk_group_create(C.byref(cfg), _ptr(devs), devs.shape[0], dir_groups, C.byref(self._g))
        if rc != 0:
            raise BflkError(rc, self._L.bflk_last_error(None).decode() or "bflk_group_create failed (NCCL missing?)")
        self.n_dir = rows * columns
        self._check(self._L.bflk_group_set_tiled_geometry(self._g, origins.shape[0], _ptr(origins)))
        self._check(self._L.bflk_group_set_grid_fov(self._g, rows, columns, float(fov)))
        self._check(self._L.bflk_group_set_kernel(self._g, kernel))

    def _check(self, rc):
        if rc != 0:
            raise BflkError(rc, self._L.bflk_group_last_error(self._g).decode())

    def size(self):
        return int(self._L.bflk_group_size(self._g))

    def power_map_batch(self, stream, n_frames):
        stream = _np(stream, np.float32)
        out = np.zeros((n_frames, self.n_dir), np.float32)
        self._check(self._L.bflk_group_power_map_batch(self._g, _ptr(stream), stream.shape[1], n_frames, _ptr(out)))
        return out

    def power_map_batch_dev(self, stream_ptrs, n_samples, n_frames, power_ptrs):
        n = self.size()
        a = (C.c_void_p * n)(*stream_ptrs)
        b = (C.c_void_p * n)(*power_ptrs)
        self._check(self._L.bflk_group_power_map_batch_dev(self._g, a, n_samples, n_frames, b))
        self._check(self._L.bflk_group_synchronize(self._g))

    def close(self):
        if getattr(self, "_g", None) is not None and self._g.value:
            self._L.bflk_group_destroy(self._g)
            self._g = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
