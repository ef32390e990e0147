"""Every compiled variant of the register-tiled kernels (das_tile.cu) at the largest delta its window admits.

Which instantiation serves a grid follows from its tables.  The largest offset spread inside a 2x2 direction tile (span0)
and inside its direction pairs (span1: the two rows of a grid column, span2: the two columns of a grid row) pick the mode
and the window chunks NCH (ensure_tiles in bflk_api.cu, das_tile_geometry in das_tile.cu); warps per CTA, stage buffers
and the channel split follow from the call.  Each NCH is a generated body with one branch per delta 0 .. 2 NCH - 9.  The
two-FMA tables also carry need_last bits (some direction of the window reaches its last chunk) and, in the two-window
modes, the `same` bit (the whole tile fits window A).  An off-by-one in any of these gives wrong samples for some
directions only, and nothing else notices.

variant_lut builds a caller LUT for which the library picks a chosen mode and NCH, with every delta 0 .. span in every
slot, windows that start at both parities of the staged rows, and both states of need_last and same.  The CPU test checks
that against a restatement of the table builder.  The GPU tests run each variant in every CTA shape it is compiled for,
hold every map to power_ref (1e-4 relative), and hold the shapes to each other bit for bit (the channel
split re-associates the channel sum, so it only meets the bar)."""
from typing import NamedTuple, Optional, Tuple

import numpy as np
import pytest

from test_batch_limits import ERR_STATE, dev_maps, power_ref, ragged_mask, rel_err

POWER_RTOL = 1e-4
R_DELAY = 20          # offsets lie in [H - R_DELAY, H]: a delay spread like a small array's, so four stage buffers fit
B = 7                 # frames per batch: an odd count leaves the last block pair half empty
SMEM_MAX = 227 * 1024
NEXT_BELOW_1 = np.nextafter(np.float32(1.0), np.float32(0.0))
ENV = ("BFLK_TILE_WARPS", "BFLK_TILE_STAGES", "BFLK_TILE_NCH", "BFLK_TILE_PAIRS", "BFLK_TILE_MODE", "BFLK_NO_KSPLIT",
       "BFLK_LAT_WARPS", "BFLK_LAT_SPLIT")


class Case(NamedTuple):
    name: str
    kernel: int                 # 2 exact form, 4 two-FMA form, 0 automatic
    spans: Tuple[int, int, int]  # (span0, span1, span2) of the table
    mode: int                   # the mode the library must pick
    nch: Optional[int]          # the window chunks it must pick (None: not tiled)
    rows: int = 6
    cols: int = 8
    H: int = 256
    N: int = 256
    dirs: Optional[Tuple[int, int]] = None   # direction range (first, count); None: the whole grid
    C: int = 96
    ragged: bool = True         # channel mask without every seventh channel


# Mode 0 at span S > 3 keeps both pair spans above the switch to two windows (>= 4, and >= 6 for S > 7); the spans of the
# other modes differ from S, so a wrong mode shows in kernel_info.  Two-window cases keep span0 above the switch.  The
# spans just below a top delta (even spans in the two-FMA form) put need_last exactly at its threshold.
CASES = [
    Case("k4-m0-s1", 4, (1, 1, 1), 0, 5),
    Case("k4-m0-s2", 4, (2, 1, 2), 0, 6, H=201),
    Case("k4-m0-s3", 4, (3, 1, 2), 0, 6, C=64, ragged=False),
    Case("k4-m0-s4", 4, (4, 4, 4), 0, 7, H=201),
    Case("k4-m0-s5", 4, (5, 4, 4), 0, 7, N=512),
    Case("k4-m0-s6", 4, (6, 4, 5), 0, 8, H=201),
    Case("k4-m0-s7", 4, (7, 4, 5), 0, 8, C=128),
    Case("k4-m0-s7-odd-grid", 4, (7, 4, 5), 0, 8, rows=5, cols=7, H=201),
    Case("k4-m0-s8", 4, (8, 6, 7), 0, 9, H=201),
    Case("k4-m0-s9-range", 4, (9, 6, 7), 0, 9, dirs=(19, 20)),
    Case("k4-m0-s10", 4, (10, 6, 7), 0, 10, H=201),
    Case("k4-m0-s11", 4, (11, 6, 7), 0, 10),
    Case("k4-m1-p2", 4, (6, 2, 4), 1, 6, H=201),
    Case("k4-m1-p3", 4, (7, 3, 5), 1, 6, C=64, ragged=False),
    Case("k4-m1-p3-tie", 4, (6, 3, 3), 1, 6),
    Case("k4-m1-p5", 4, (9, 5, 7), 1, 7, H=201, N=512),
    Case("k4-m2-p3", 4, (7, 5, 3), 2, 6, H=201, N=512),
    Case("k4-m2-p4", 4, (9, 6, 4), 2, 7),
    Case("k4-m2-p5-range", 4, (9, 7, 5), 2, 7, dirs=(11, 30)),
    Case("k2-m0-s1", 2, (1, 1, 1), 0, 5, H=201),
    Case("k2-m0-s2", 2, (2, 1, 2), 0, 6),
    Case("k2-m0-s3", 2, (3, 1, 2), 0, 6, H=201),
    Case("k2-m0-s4", 2, (4, 4, 4), 0, 7, C=64, ragged=False),
    Case("k2-m0-s5", 2, (5, 4, 4), 0, 7, H=201),
    Case("k2-m0-s6", 2, (6, 4, 5), 0, 8),
    Case("k2-m0-s7-range", 2, (7, 4, 5), 0, 8, H=201, dirs=(19, 20)),
    Case("k2-m0-s10", 2, (10, 6, 7), 0, 10),
    Case("k2-m0-s11", 2, (11, 6, 7), 0, 10, H=201, N=512),
    Case("k2-m1-p3-range", 2, (7, 3, 5), 1, 6, H=201, dirs=(11, 30)),
    Case("k2-m1-p5", 2, (9, 5, 7), 1, 7, C=128, ragged=False),
    Case("k2-m1-p5-tie", 2, (9, 5, 5), 1, 7),
    Case("k2-m2-p3-odd-grid", 2, (7, 5, 3), 2, 6, rows=5, cols=7),
    Case("k2-m2-p5", 2, (9, 7, 5), 2, 7, H=201),
]
BOUNDARY = [
    Case("k0-m0-s11", 0, (11, 6, 7), 0, 10),
    Case("k0-m0-s12", 0, (12, 6, 7), 0, None, H=201),
]


# ---- restatement of the table builder (no GPU) ----------------------------------------------------------------------------
def tile_offsets(off, rows, cols, first, count, index, mode):
    """Offsets [tile][usable channel][slot] as build_tiles_kernel reads them (tables.cu:98-126): tiles over the grid rows
    the direction range touches, slots in window order (mode 1: the two rows of a grid column share a window), and a
    direction missing at an odd grid's edge aliasing the tile's first existing direction (tables.cu:107-111).  Also the
    range-local direction of every (tile, slot), -1 where it is not stored."""
    row0, row1 = (first // cols) & ~1, (first + count - 1) // cols
    tile_cols = (cols + 1) // 2
    n_tiles = ((row1 - row0) // 2 + 1) * tile_cols
    dirs = np.full((n_tiles, 4), -1, np.int64)
    for t in range(n_tiles):
        tr, tc = divmod(t, tile_cols)
        for slot in range(4):
            q = ((slot & 1) << 1 | slot >> 1) if mode == 1 else slot
            r, c = row0 + 2 * tr + (q >> 1), 2 * tc + (q & 1)
            if r < rows and c < cols:
                dirs[t, slot] = r * cols + c
    ref = np.array([next(g for g in d if g >= 0) for d in dirs])
    g = np.where(dirs >= 0, dirs, ref[:, None])
    o = off[g][:, :, index].transpose(0, 2, 1).astype(np.int64)
    local = np.where((dirs >= first) & (dirs < first + count), dirs - first, -1)
    return o, local


def table_entries(o, mode, pair_span, stage_off):
    """What build_tiles_kernel stores per (tile, channel) entry (tables.cu:127-165): deltas [..][slot], span, the parity
    of each window's start relative to the staged rows [..][window], need_last [..][window] (bits 29 / 30) and same."""
    if mode == 0:
        base = o.min(-1)
        d = o - base[..., None]
        span = d.max(-1)
        odd = np.stack([(base - stage_off) & 1] * 2, -1)
        need = np.stack([span >= pair_span - 1, np.zeros_like(span, bool)], -1)
        same = np.zeros(span.shape, bool)
    else:
        lo4, hi4 = o.min(-1), o.max(-1)
        same = hi4 - lo4 <= pair_span
        base = np.stack([np.where(same, lo4, np.minimum(o[..., 0], o[..., 1])),
                         np.where(same, lo4, np.minimum(o[..., 2], o[..., 3]))], -1)
        d = o - np.repeat(base, 2, axis=-1)
        span = d.max(-1)
        odd = (base - stage_off) & 1
        hit = d >= pair_span - 1
        need_a, need_b = hit[..., 0] | hit[..., 1], hit[..., 2] | hit[..., 3]
        need = np.stack([need_a | (same & need_b), ~same & need_b], -1)
    return dict(deltas=d, span=span, odd=odd, need_last=need, same=same)


def table_spans(off, rows, cols, first, count, index):
    """(span0, span1, span2): pass 1 of ensure_tiles, the builder run with pair_span -1 (bflk_api.cu:502-511)."""
    return tuple(int(table_entries(tile_offsets(off, rows, cols, first, count, index, m)[0], m, -1, 0)["span"].max())
                 for m in range(3))


def choose_mode(spans):
    """bflk_api.cu:516-519: two windows when the tile spread is too wide for one and the direction pairs fit."""
    pair, pair_mode = min(spans[1], spans[2]), 1 if spans[1] <= spans[2] else 2
    if (spans[0] > 3 and pair <= 3) or (spans[0] > 7 and pair <= 5):
        return pair_mode
    return 0


def window_chunks(span, mode, fast):
    """das_tile.cu:446-448: NCH of the exact and the two-FMA form."""
    if fast:
        return max(6 if mode else 5, (9 + span + 1) // 2)
    return 5 if span <= 1 and mode == 0 else 6 if span <= 3 else 7 if span <= 5 else 8 if span <= 7 else 10


def compiled_warps(nch, mode, fast):
    """The warps per CTA kTileVariants lists for the variant (das_tile.cu:392-414), each reachable with BFLK_TILE_WARPS
    (das_tile.cu:461): 16 too for the exact form at NCH >= 7, which the automatic choice never gives,
    except the exact two-window NCH 7, compiled for 10 - 12 warps only."""
    return (10, 11, 12) if not fast and mode != 0 and nch == 7 else (10, 11, 12, 16)


def smem_bytes(H, stage_off, nch, mode, fast, warps, stages):
    """das_tile_smem_bytes with the packed-row size of das_tile_geometry (das_tile.cu:434-438, 463-465)."""
    last = (H - stage_off) // 2 + 4 * 31 + nch - 1
    row_bytes = 2 * 16 * (last + last // 4 + 1)
    entry = (80 if mode else 64) if fast else 32
    return stages * (8 * row_bytes + warps * 8 * entry) + stages * 12 + 256


# ---- the table generator (no GPU) -------------------------------------------------------------------------------------------
def pattern(kind, k, v, case):
    """Offsets above the entry's base at grid positions q = 2 * row + col of a tile (slot order of modes 0 and 2).
    "tile": position k at v, its diagonal at 0, its column and row neighbours as low as span1 / span2 allow (v <= span0
    <= span1 + span2 keeps every spread within the case's spans).  "pair" (two-window modes): k at v and its pair mate at
    0 in one window, the same two raised by as much as the span across the pairs allows in the other window, so that
    most such tiles do not fit one window (`same` clear)."""
    s0, s1, s2 = case.spans
    d = np.zeros(4, np.int64)
    d[k] = v
    if kind == "tile":
        d[k ^ 2] = max(0, v - s1)
        d[k ^ 1] = max(0, v - s2)
    else:
        mate, across, q = (k ^ 1, 2, s1) if case.mode == 2 else (k ^ 2, 1, s2)
        lift = min(q, s0 - v)
        d[k ^ across] = v + lift
        d[mate ^ across] = lift
    return d


def variant_lut(case, seed=0):
    """Caller LUT off, frac [rows * cols][C] and channel mask for a case.  Entry (tile t, usable channel s) takes pattern
    (s + 7 t) mod n of the n (kind, position, delta, parity) combinations, on a random base of that parity in
    [H - R_DELAY, H - span0].  Tiles at an odd grid's edge get a random pair within min(span1, span2)."""
    rng = np.random.default_rng(seed)
    rows, cols, C, H = case.rows, case.cols, case.C, case.H
    s0, s1, s2 = case.spans
    P = case.spans[case.mode]
    combos = [("tile", k, v, p) for k in range(4) for v in range(s0 + 1) for p in (0, 1)]
    if case.mode:
        combos += [("pair", k, v, p) for k in range(4) for v in range(P + 1) for p in (0, 1)]
    index = ragged_mask(C) if case.ragged else np.arange(C, dtype=np.int32)
    pos = np.full(C, -1)
    pos[index] = np.arange(len(index))
    lo, hi = H - R_DELAY, H - s0
    near = min(s1, s2)
    off = np.zeros((rows * cols, C), np.int64)
    tile_cols = (cols + 1) // 2
    for t in range(((rows + 1) // 2) * tile_cols):
        tr, tc = divmod(t, tile_cols)
        qs = [q for q in range(4) if 2 * tr + (q >> 1) < rows and 2 * tc + (q & 1) < cols]
        dirs = [(2 * tr + (q >> 1)) * cols + 2 * tc + (q & 1) for q in qs]
        for c in range(C):
            if len(qs) < 4:
                d = np.zeros(4, np.int64)
                d[qs[1:]] = rng.integers(-near, near + 1, len(qs) - 1)
                d -= d[qs].min()
                p = int(rng.integers(2))
            else:
                i = pos[c] if pos[c] >= 0 else int(rng.integers(len(combos)))
                kind, k, v, p = combos[(i + 7 * t) % len(combos)]
                d = pattern(kind, k, v, case)
            base = int(rng.integers(lo, hi + 1))
            if base % 2 != p:
                base += 1 if base < hi else -1
            off[dirs, c] = base + d[qs]
    frac = rng.random(off.shape, dtype=np.float32)
    frac[::7] = 0.0
    frac[3::7] = NEXT_BELOW_1
    frac[:, 5] = 0.0
    frac[:, 6] = NEXT_BELOW_1
    return off.astype(np.int32), frac, index


def dir_range(case):
    return case.dirs or (0, case.rows * case.cols)


def stage_origin(off):
    """(H - max_delay) & ~1 with max_delay = H - the LUT's smallest offset (bflk_api.cu:287, das_tile.cu:444)."""
    return int(off.min()) & ~1


@pytest.mark.parametrize("case", CASES + BOUNDARY, ids=lambda c: c.name)
def test_generator_hits_variant(case):
    off, frac, index = variant_lut(case)
    first, count = dir_range(case)
    assert off.min() >= case.H - R_DELAY and off.max() <= case.H
    assert frac.min() >= 0.0 and frac.max() == NEXT_BELOW_1 and (frac == 0.0).any()
    spans = table_spans(off, case.rows, case.cols, first, count, index)
    assert spans == case.spans
    mode = choose_mode(spans)
    assert mode == case.mode
    S = spans[mode]
    if case.nch is None:
        assert S > 11                       # das_tile_max_span
        return
    fast = case.kernel != 2
    nch = window_chunks(S, mode, fast)
    assert nch == case.nch
    top = 2 * nch - 9                       # the largest delta of the NCH body (bflk_api.cu:540)
    assert S <= top <= S + 1
    stage_off = stage_origin(off)
    o, _ = tile_offsets(off, case.rows, case.cols, first, count, index, mode)
    e = table_entries(o, mode, top, stage_off)
    d = e["deltas"]
    assert d.min() == 0 and d.max() <= top
    # every delta of the body in every slot, from windows that start at both parities of the staged rows
    for slot in range(4):
        win = np.where(e["same"], 0, slot >> 1)
        odd = np.take_along_axis(e["odd"], win[..., None], -1)[..., 0]
        for v in range(S + 1):
            for p in (0, 1):
                assert ((d[..., slot] == v) & (odd == p)).any(), (slot, v, p)
    # entries in which a single slot reaches the case's largest delta
    assert ((d == S).sum(-1) == 1).any()
    if fast:
        need = e["need_last"]
        if nch == 5:
            assert need[..., 0].all()       # threshold 0: the last chunk is always read
        else:
            assert need.any() and (~need[..., 0]).any()
    if mode:
        same = e["same"]
        assert same.any() and (~same).any()
        for slot in range(4):
            for v in range(S + 1):
                assert ((d[~same][:, slot]) == v).any(), (slot, v)
    # four stage buffers fit in every throughput shape the variant runs, so BFLK_TILE_STAGES=4 is not cut to 3
    for warps in compiled_warps(nch, mode, fast):
        assert smem_bytes(case.H, stage_off, nch, mode, fast, warps, 4) <= SMEM_MAX


def test_restated_choice_matches_the_issue_thresholds():
    """NCH per span of each form, and the 12-chunk wall (das_tile.cu:446-448, das_tile_max_span)."""
    assert [window_chunks(s, 0, True) for s in range(12)] == [5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10]
    assert [window_chunks(s, 0, False) for s in range(12)] == [5, 5, 6, 6, 7, 7, 8, 8, 10, 10, 10, 10]
    assert [window_chunks(s, m, f) for m in (1, 2) for f in (False, True) for s in (0, 3, 4, 5)] == [6, 6, 7, 7] * 4
    assert choose_mode((4, 3, 4)) == 1 and choose_mode((4, 4, 3)) == 2 and choose_mode((4, 3, 3)) == 1
    assert choose_mode((8, 5, 6)) == 1 and choose_mode((8, 6, 6)) == 0 and choose_mode((7, 4, 4)) == 0


# ---- the variant matrix (GPU) -----------------------------------------------------------------------------------------------
def white_noise(case, seed=1):
    """[C][T] float32 white noise, T the least even length that holds B frames; host copy and device copy."""
    import torch
    T = (B - 1) * case.N + case.H + case.N + 1
    T += T & 1
    x = np.random.default_rng(seed).standard_normal((case.C, T)).astype(np.float32)
    return x, torch.from_numpy(x).cuda()


def make_beamformer(case, off, frac, index, monkeypatch, env):
    """A handle for the case's LUT with the BFLK_* settings `env` (read once, by the constructor)."""
    import bflk
    with monkeypatch.context() as m:
        for k in ENV:
            m.delenv(k, raising=False)
        for k, v in env.items():
            m.setenv(k, str(v))
        w = bflk.Beamformer(n_channels=case.C, frame_len=case.N, history=case.H, window_len=case.H + case.N + 1)
    w.set_geometry(np.zeros((case.C, 3), np.float32))
    w.set_grid_tables(off, frac)
    w.set_grid_shape(case.rows, case.cols)
    w.set_channel_mask(index)
    if case.dirs:
        w.set_direction_range(*case.dirs)
    w.set_kernel(case.kernel)
    return w


def assert_near(p, ref, what):
    assert np.all(np.isfinite(p)), what
    assert rel_err(p, ref) <= POWER_RTOL, (what, rel_err(p, ref))


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=lambda c: c.name)
def test_variant(case, monkeypatch):
    """The throughput shape (every warps count the variant is compiled for, 3 and 4 stage buffers, through _dev_submit /
    _dev_join and power_map_batch_dev), the latency shape (power_map_batch_dev of B frames and of single frames) and, in the
    two-FMA form, single frames with the channels split over clusters of 2 and 4 CTAs."""
    import bflk
    off, frac, index = variant_lut(case)
    first, count = dir_range(case)
    x_host, x = white_noise(case)
    ref = power_ref(x_host, off[first:first + count], frac[first:first + count], index, case.N, range(B))
    info = (case.kernel, case.spans[case.mode], case.nch)
    fast = case.kernel == 4
    single = {b: x[:, b * case.N:].contiguous() for b in (0, B - 1)}

    # automatic CTA shape: the throughput tables for _dev_submit, the latency shape for the batch and single frames
    assert bflk.launch_shape(case.rows, case.cols, len(index), B, case.N)[0] > 0
    w = make_beamformer(case, off, frac, index, monkeypatch, {})
    want = dev_maps(w, x, B, submit=True)
    assert w.kernel_info() == info
    for b in range(B):
        assert_near(want[b], ref[b], (case.name, "throughput", b))
    assert np.array_equal(dev_maps(w, x, B), want), "latency shape"
    assert w.kernel_info() == info
    for b, xb in single.items():
        assert np.array_equal(dev_maps(w, xb, 1)[0], want[b]), ("single frame", b)
    w.close()

    for warps in compiled_warps(case.nch, case.mode, fast):
        for stages in (3, 4):
            w = make_beamformer(case, off, frac, index, monkeypatch, {"BFLK_TILE_WARPS": warps, "BFLK_TILE_STAGES": stages})
            assert np.array_equal(dev_maps(w, x, B, submit=True), want), (warps, stages, "submit")
            assert w.kernel_info() == info
            assert np.array_equal(dev_maps(w, x, B), want), (warps, stages, "batch")
            w.close()

    if fast:
        for split in (None, 2, 4):
            w = make_beamformer(case, off, frac, index, monkeypatch, {"BFLK_LAT_SPLIT": split} if split else {})
            w.set_channel_split(True)
            for b, xb in single.items():
                assert_near(dev_maps(w, xb, 1)[0], ref[b], (case.name, "split", split, b))
                assert w.kernel_info() == info
            w.close()


@pytest.mark.gpu
def test_span_12_is_not_tiled(monkeypatch):
    """Span 11 is the widest window (NCH 10); at 12 the automatic choice falls back to the lane-broadcast kernel and still
    meets the bar, and an explicit register-tiled kernel refuses the call."""
    import bflk
    for case in BOUNDARY:
        off, frac, index = variant_lut(case)
        x_host, x = white_noise(case)
        ref = power_ref(x_host, off, frac, index, case.N, range(B))
        w = make_beamformer(case, off, frac, index, monkeypatch, {})
        got = dev_maps(w, x, B)
        if case.nch is None:
            assert w.kernel_info() == (3, case.spans[0], 0)
        else:
            assert w.kernel_info() == (4, case.spans[0], case.nch)
        for b in range(B):
            assert_near(got[b], ref[b], (case.name, b))
        if case.nch is None:
            for kernel in (2, 4):
                w.set_kernel(kernel)
                with pytest.raises(bflk.BflkError) as e:
                    dev_maps(w, x, B)
                assert e.value.code == ERR_STATE, (kernel, str(e.value))
        w.close()
