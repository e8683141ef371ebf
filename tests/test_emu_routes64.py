"""The kernel source on the CPU SIMT emulator (tests/emu) against the float64 reference (tests/ref64.py), with the inputs of
tests/test_gpu_routes64.py: levels from 1 down to 3e-7 with silent and subnormal stretches inside the streams, a cosine
at every bin, a unit impulse at every frame offset, the stereo identities and loud inputs, at power_scale 1 and 1 / N^2.

The emulator runs the product's .cuh files with libm in place of MUFU.LG2 and fma in place of FFMA2; this half fixes the
calibration of ref64.A and ref64.B_REL where no GPU is present.  Also here: the pin of ref64 to the oracle under the
north-star criterion of tests/parity.py, so that the float64 reference cannot drift from the reference semantics."""
import numpy as np
import pytest

import emu_lib as E
import oracle_lib as O
import parity
import ref64
import signals
from jadespectrogram_b200._capi import MIX, ROWS, WIN, JadeConfig

pytestmark = pytest.mark.timeout(300)


def _cfg(N, hop, ch, window="hann", mix="absmean", **kw):
    c = JadeConfig()
    c.sample_rate = 48000.0
    c.fft_size, c.hop, c.frames_per_block, c.block_stride, c.preroll = N, hop, 1, hop, -1
    c.window, c.channels, c.mix_mode = WIN[window], ch, MIX[mix]
    c.row_map, c.flip_y, c.power_scale = 0, 1, 1.0
    for k, v in kw.items():
        setattr(c, k, v)
    return c


@pytest.mark.parametrize("N,hop,ch,window,mix,kw", [
    (64, 16, 1, "rect", "absmean", {}), (256, 64, 3, "flattop", "min", {}), (1024, 205, 2, "hannpoisson", "max", {}),
    (2048, 512, 2, "hann", "absmean", {}), (512, 128, 2, "hann", "right", {}),
    (4096, 1024, 2, "blackmanharris", "absmean", dict(frames_per_block=2, block_stride=2048, preroll=1000))])
def test_ref64_matches_oracle(N, hop, ch, window, mix, kw):
    """ref64 and the oracle agree under parity.check_db, both ways round (the oracle only knows preroll = N, one frame per
    block: the last geometry is compared with frames re-based to that layout)."""
    c = _cfg(N, hop, ch, window, mix, **kw)
    x = signals.streams(1, ch, hop * 24 + 64, 48000.0)[0]
    x[:, hop * 8:hop * 8 + N + hop] *= 1e-4
    ncols, j0 = 21, (4 if kw else 0)
    r = ref64.Ref(c, x, j0, ncols)
    # frame j of the last geometry starts at (j // 2) * 2048 + (j % 2) * 1024 - 1000 == j * 1024 - 1000: the oracle's frame
    # j * 1024 - 4096 over the samples from 3096 on, for the columns whose frames start at or after sample 0 of that view
    xo = x[:, N - 1000:] if kw else x
    odb, _ = O.render_batch(xo, fft_size=N, hop=hop, window=window, mix=mix, first_col=j0, ncols=ncols)
    parity.check_db(r.db.astype(np.float32), odb, N, "ref64 vs oracle")
    parity.check_db(odb, r.db.astype(np.float32), N, "oracle vs ref64")


def test_ref64_mix_semantics():
    """Max starts at 0, Min at 1e6 (a channel louder than 1e6 in every bin shows 60 dB), Left / Right pick a channel."""
    pc = np.array([[[4.0, 2e6, 0.0], [1.0, 3e6, 5.0]]])
    for mix, want in (("absmean", [2.5, 2.5e6, 2.5]), ("max", [4.0, 3e6, 5.0]), ("min", [1.0, 1e6, 0.0]),
                      ("left", [4.0, 2e6, 0.0]), ("right", [1.0, 3e6, 5.0])):
        p, _ = ref64.mix(_cfg(4, 1, 2, mix=mix), pc)
        assert np.array_equal(p[0], want), mix
    assert ref64.SILENT_DB == np.float32(-110.0)


def _check(c, x, grid=2, want_db=True, ncols=None, rng=(-50.0, 50.0)):
    """Render x [streams][ch][n] on the emulator and compare every stream with ref64; returns the worst db_errors."""
    N, hop = c.fft_size, c.hop
    ncols = ncols or x.shape[2] // hop + 1
    pal = O.Palette(256, O.PAL["jade"])
    db, pix = E.render(c, pal.table(), rng[0], rng[1], x, 0, ncols, len(ref64.row_bins(c)[0]), grid=grid, want_db=want_db)
    worst = dict(frac=0.0, a=0.0, b=0.0, ddb=0.0)
    for s in range(x.shape[0]):
        r = ref64.Ref(c, x[s], 0, ncols)
        if want_db:
            e = ref64.check_db64(db[s], r, f"stream {s}")
            worst = {k: max(worst[k], e[k]) for k in worst}
        ref64.check_pixels64(pix[s], r, pal, rng[0], rng[1], 256, f"stream {s}")
    return worst, db, pix


def _inputs(ch, N, hop, kinds=None):
    kinds = kinds or ref64.standard_kinds(ch, N, hop)
    n = ref64.stream_length(N, hop, -(-len(ref64.impulse_offsets(N, hop)) // 8))
    return ref64.batch(kinds, ch, N, hop, n)


@pytest.mark.parametrize("N,ch", [(128, 1), (128, 2), (256, 4), (512, 1), (1024, 2)])
@pytest.mark.parametrize("ps", [1.0, "1/N^2"])
def test_emulated_pksmall_float64(monkeypatch, N, ch, ps):
    """pksmall<T>: staged instantiations (dB-storing and pixel-only) and the guarded one render the same columns; both
    within the float64 bound on every input family."""
    monkeypatch.delenv("JADE_EMU_FORCE_GUARD", raising=False)
    hop = N // 4
    c = _cfg(N, hop, ch, power_scale=1.0 if ps == 1.0 else float(np.float32(1.0 / N ** 2)))
    x = _inputs(ch, N, hop)
    _, db, pix = _check(c, x)
    _check(c, x, want_db=False)
    monkeypatch.setenv("JADE_EMU_FORCE_GUARD", "1")
    _, gdb, gpix = _check(c, x)
    assert np.array_equal(gdb, db) and np.array_equal(gpix, pix)


@pytest.mark.parametrize("hop", [256, 512])
def test_emulated_pk2048_mono_float64(monkeypatch, hop):
    """pk2048, one channel: cp.async staging (dB and pixel-only), the ring instantiation of the hop (RING4 / RING8, dB and
    pixel-only), power_scale 1 and 1 / N^2."""
    for k in ("JADE_EMU_FORCE_GUARD", "JADE_EMU_RING", "JADE_EMU_NOPAIR", "JADE_EMU_PAIR2"):
        monkeypatch.delenv(k, raising=False)
    N = 2048
    kinds = ref64.standard_kinds(1, N, hop)
    x = _inputs(1, N, hop, [k for k in kinds if k[0] != "impulse"] + [("impulse", i) for i in (0, 3)])
    for ps in (1.0, float(np.float32(1.0 / N ** 2))):
        c = _cfg(N, hop, 1, power_scale=ps)
        _, db, pix = _check(c, x, grid=4)
        _check(c, x, grid=4, want_db=False)
        monkeypatch.setenv("JADE_EMU_RING", "1")
        _, rdb, rpix = _check(c, x, grid=4)
        _check(c, x, grid=4, want_db=False)
        monkeypatch.delenv("JADE_EMU_RING")
        assert np.array_equal(rdb, db) and np.array_equal(rpix, pix)


def test_emulated_pkz2048_float64(monkeypatch):
    """pkz2048 (two channels as one complex transform): staged, guarded and ring instantiations, dB-storing, pixel-only
    and u8, over the stereo identities (one channel silent, L = R, L = -R, R = 1e-6 L) and the other families."""
    for k in ("JADE_EMU_FORCE_GUARD", "JADE_EMU_RING", "JADE_EMU_NOPAIR", "JADE_EMU_PAIR2"):
        monkeypatch.delenv(k, raising=False)
    N, hop = 2048, 512
    kinds = ref64.standard_kinds(2, N, hop)
    x = _inputs(2, N, hop, [k for k in kinds if k[0] != "impulse"] + [("impulse", i) for i in (1, 6)])
    for ps in (1.0, float(np.float32(1.0 / N ** 2))):
        c = _cfg(N, hop, 2, power_scale=ps)
        _, db, pix = _check(c, x, grid=4)
        for rng in ((-50.0, 50.0), (-120.0, 60.0), (58.0, 59.0)):
            _check(c, x, grid=4, want_db=False, rng=rng)
        monkeypatch.setenv("JADE_EMU_RING", "1")
        _, rdb, rpix = _check(c, x, grid=4)
        _check(c, x, grid=4, want_db=False)
        monkeypatch.delenv("JADE_EMU_RING")
        monkeypatch.setenv("JADE_EMU_FORCE_GUARD", "1")
        _, gdb, gpix = _check(c, x, grid=4)
        monkeypatch.delenv("JADE_EMU_FORCE_GUARD")
        assert np.array_equal(rdb, db) and np.array_equal(gdb, db)


@pytest.mark.parametrize("N,ch,mix,kw", [
    (4096, 1, "absmean", {}), (8192, 2, "absmean", {}), (16384, 1, "absmean", {}),
    (4096, 2, "min", {}), (8192, 1, "absmean", dict(db_precise=1)), (4096, 1, "absmean", dict(flip_y=0)), (4096, 3, "absmean", {}),
    (1024, 2, "max", {}), (512, 1, "absmean", dict(db_precise=1, flip_y=0)), (256, 3, "absmean", {}),
    (1024, 1, "absmean", dict(row_map=ROWS["linear_crop"], fmin=1000.0, fmax=8000.0)),
    (2048, 1, "absmean", dict(row_map=ROWS["log_maxpool"], rows=64, fmin=50.0, fmax=20000.0))])
def test_emulated_cta_warp_pk3_float64(N, ch, mix, kw):
    """pkcta<R1>, pk3<16384> and the general warp / cta kernels (precise dB, un-flipped, crop, log rows, Max / Min, three
    channels): levels, a comb of bins, impulses."""
    hop = N // 4
    kinds = [("level", i) for i in range(5)] + [("bins", i) for i in (0, 5)] + [("impulse", i) for i in (2,)] + [("loud", 0)]
    x = _inputs(ch, N, hop, kinds)[:, :, :12 * N]
    c = _cfg(N, hop, ch, mix=mix, **kw)
    _check(c, x, grid=3)


def test_emulated_pkcl65536_stereo_float64(monkeypatch):
    """N = 65536, two channels (pkcl65536): AbsMean and Max over silent, equal and opposite channels."""
    monkeypatch.delenv("JADE_EMU_CTA2", raising=False)
    monkeypatch.delenv("JADE_EMU_PKCL", raising=False)
    N, hop = 65536, 32768
    kinds = [("stereo", 0), ("stereo", 2), ("stereo", 3), ("level", 3)]
    x = ref64.batch(kinds, 2, N, hop, 6 * N)
    for mix in ("absmean", "max"):
        _check(_cfg(N, hop, 2, mix=mix), x, grid=2)
