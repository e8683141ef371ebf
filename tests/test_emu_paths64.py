"""The kernel source on the CPU SIMT emulator (tests/emu) against the float64 reference (tests/ref64.py), on the paths of
tests/test_gpu_paths64.py that the emulator takes too: block geometries (feed 10 % and 25 %, three frames per block that
are not evenly spaced, pre-roll 0, odd and 3 N + 2, hop 3 N / 2), Left / Right on two and three channels (the long-run
N = 2048 form included, across stream changes) and column windows starting after column 0 or running past the end.

The emulator takes the configuration as given (three frames per block run the division form of frame_start; the engine
folds evenly spaced geometries into one frame per block) and routes columns the way launch_stft does."""
import numpy as np
import pytest

import emu_lib as E
import oracle_lib as O
import ref64
from jadespectrogram_b200._capi import MIX, ROWS, WIN, JadeConfig

pytestmark = pytest.mark.timeout(600)

GEOMS = {"feed10": lambda N: (int(0.1 * N + 0.5), 10, N, N), "feed25": lambda N: (N // 4, 4, N, N),
         "fb3": lambda N: (N // 4, 3, N, N), "preroll0": lambda N: (N // 4, 1, N // 4, 0),
         "preroll_odd": lambda N: (N // 4, 1, N // 4, N // 2 + 3), "preroll3N+2": lambda N: (N // 4, 1, N // 4, 3 * N + 2),
         "hop3N/2": lambda N: (3 * N // 2, 1, 3 * N // 2, N)}
# (N, channels, mix, extra configuration): the packed kernels of each size, pkz2048, pkcta<2> and the general warp / cta
FAMILIES = [(128, 1, "absmean", {}), (256, 2, "absmean", {}), (1024, 1, "absmean", {}), (2048, 1, "absmean", {}),
            (2048, 2, "absmean", {}), (4096, 1, "absmean", {}), (512, 1, "absmean", dict(flip_y=0)),
            (4096, 2, "max", {})]


def _cfg(N, ch, mix="absmean", geom=None, **kw):
    hop, fb, stride, preroll = geom if geom else (N // 4, 1, N // 4, N)
    c = JadeConfig()
    c.sample_rate = 48000.0
    c.fft_size, c.hop, c.frames_per_block, c.block_stride, c.preroll = N, hop, fb, stride, preroll
    c.window, c.channels, c.mix_mode = WIN["hann"], ch, MIX[mix]
    c.row_map, c.flip_y, c.power_scale = ROWS["identity"], 1, 1.0
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def _columns(c, n):
    """Columns whose frame ends inside n samples (jade_columns_for in hop mode)."""
    N = c.fft_size
    j = 0
    while ref64.frame_starts(c, j, 1)[0] + N <= n:
        j += 1
    return j


def _inputs(ch, N, hop):
    kinds = [("level", 0), ("level", 4), ("bins", 3), ("impulse", 1), ("loud", 0)] + ([("stereo", 3)] if ch > 1 else [])
    n = ref64.stream_length(N, hop, 2)
    return ref64.batch(kinds, ch, N, hop, n)


def _check(c, x, first, ncols, grid=3):
    """Render columns [first, first + ncols) of x on the emulator (dB-storing and pixel-only) and compare every stream
    with ref64."""
    pal = O.Palette(256, O.PAL["jade"])
    R = len(ref64.row_bins(c)[0])
    db, pix = E.render(c, pal.table(), -50.0, 50.0, x, first, ncols, R, grid=grid, want_db=True)
    _, pix2 = E.render(c, pal.table(), -50.0, 50.0, x, first, ncols, R, grid=grid, want_db=False)
    for s in range(x.shape[0]):
        r = ref64.Ref(c, x[s], first, ncols)
        ref64.check_db64(db[s], r, f"stream {s}")
        ref64.check_pixels64(pix[s], r, pal, -50.0, 50.0, 256, f"stream {s}")
        ref64.check_pixels64(pix2[s], r, pal, -50.0, 50.0, 256, f"stream {s} pixel-only")


@pytest.fixture(autouse=True)
def _product_routes(monkeypatch):
    for k in ("JADE_EMU_FORCE_GUARD", "JADE_EMU_RING", "JADE_EMU_NOPAIR", "JADE_EMU_PAIR2", "JADE_EMU_CTA2", "JADE_EMU_PKCL",
              "JADE_EMU_PKCTA", "JADE_EMU_NO_U8"):
        monkeypatch.delenv(k, raising=False)


@pytest.mark.parametrize("geom", list(GEOMS))
@pytest.mark.parametrize("N,ch,mix,kw", FAMILIES)
def test_emulated_geometry_float64(N, ch, mix, kw, geom):
    """Every column of a stream under each block geometry."""
    c = _cfg(N, ch, mix, GEOMS[geom](N), **kw)
    x = _inputs(ch, N, max(1, c.block_stride // c.frames_per_block))
    _check(c, x, 0, _columns(c, x.shape[2]))


@pytest.mark.parametrize("N,kw", [(256, {}), (1024, {}), (2048, {}), (4096, {}), (512, dict(flip_y=0))])
@pytest.mark.parametrize("mix", ["left", "right"])
@pytest.mark.parametrize("ch", [2, 3])
def test_emulated_channel_select_float64(N, kw, mix, ch):
    """Left / Right read channel 0 / 1 of a multi-channel stream (channel_range), aligned and odd geometries."""
    for geom in (None, GEOMS["feed10"](N)):
        c = _cfg(N, ch, mix, geom, **kw)
        x = _inputs(ch, N, c.hop)
        _check(c, x, 0, _columns(c, x.shape[2]))


@pytest.mark.parametrize("hop", [256, 512])
def test_emulated_long_run_right_after_column_0(monkeypatch, hop):
    """The long-run N = 2048 form (tensor-memory sample ring) with Right on two channels, from column 3: each warp walks
    a contiguous run of columns over several streams and restarts at the window's first column on every stream change."""
    monkeypatch.setenv("JADE_EMU_RING", "1")
    N = 2048
    c = _cfg(N, 2, "right", (hop, 1, hop, N))
    x = ref64.batch([("level", 0), ("level", 2), ("stereo", 1), ("stereo", 4), ("loud", 1)], 2, N, hop, 40 * hop)
    # interior columns only (frames inside the stream): the run form takes the whole launch
    first = N // hop + 3
    _check(c, x, first, _columns(c, x.shape[2]) - first, grid=2)


@pytest.mark.parametrize("N,ch,mix,kw", [(256, 1, "absmean", {}), (2048, 1, "absmean", {}), (2048, 2, "absmean", {}),
                                         (4096, 2, "absmean", {}), (512, 2, "min", {})])
def test_emulated_column_windows_float64(N, ch, mix, kw):
    """Windows starting at column 1, mid-stream and near the end, and windows running past the end of the stream."""
    c = _cfg(N, ch, mix, None, **kw)
    x = _inputs(ch, N, c.hop)
    total = _columns(c, x.shape[2])
    for a, n in ((1, total - 1), (total // 2, total // 4), (total - 3, 3), (total - 4, 6), (total // 3, total - total // 3 + 3)):
        _check(c, x, a, n)
