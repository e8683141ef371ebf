"""A float64 reference of the whole path (framing, window, power, channel mix, dB, row map, palette), in plain numpy.

The oracle (oracle/jade_oracle.cpp) restates the original plugin in float32 with a float32 FFT, so tests/parity.py has to
allow for float32 FFT error on both sides (1e-4 relative in magnitude).  This module carries no float32 arithmetic past the
window table, so its criterion, check_db64, can be about five times tighter:

    M = sqrt(p + 1e-11)  (p: mixed power, the quantity whose dB is shown)
    |M_gpu - M64| <= A * eps32 * sqrt(log2(N) * E64 / N) + (B_REL + DB32) * M64

E64 is the frame's energy sum(p) over its bins: for AbsMean that of the mixed power, for the other mixes that of the
loudest contributing channel (Max / Min / Left / Right pick a channel per bin; the rounding noise of a bin is set by the
energy of the channel it came from).  DB32 is the rounding of a float32 dB value (1 ulp at |dB| in [64, 128) is 7.6e-6 dB,
0.9e-6 relative in M; four ulps, as in parity.py).

Calibration of A and B_REL: the worst normalised errors of the kernels, measured on the CPU emulator (tests/emu: the same
.cuh files, libm in place of MUFU.LG2) over every input family of test_emu_routes64.py (levels from 1 down to 3e-7 with
silent and subnormal stretches, a cosine at every bin, a unit impulse at every frame offset, stereo identities, loud inputs,
power_scale 1 and 1 / N^2):
  * floor term, |M_gpu - M64| / (eps32 sqrt(log2(N) E64 / N)) on bins more than 40 dB below the frame peak:  5.6  -> A = 12
  * relative term, |M_gpu - M64| / M64 on bins within 40 dB of the frame peak:                    7.3e-6 -> B_REL = 2e-5
  * the whole bound: at most 0.35 of it used on any bin.
The oracle's float32 output, on the inputs of test_emu_routes64.py::test_ref64_matches_oracle, uses at most 0.12 of it.
"""
import ctypes as C

import numpy as np

import oracle_lib as O

EPS32 = float(np.finfo(np.float32).eps)
A = 12.0
B_REL = 2e-5
DB32 = 4e-6
FLOOR = 1e-11                                       # Spectrogram.cpp:36,107: dB = 10 log10(p + 1e-11)
SILENT_DB = np.float32(10.0 * np.log10(np.float64(np.float32(FLOOR))))

MIX_ABSMEAN, MIX_MAX, MIX_MIN, MIX_LEFT, MIX_RIGHT = range(5)
ROWS_IDENTITY, ROWS_LINEAR_CROP, ROWS_LOG_MAXPOOL = range(3)


def _geometry(cfg):
    """(N, hop, frames_per_block, block_stride, preroll) with the defaults jade_configure applies."""
    N, hop = int(cfg.fft_size), int(cfg.hop)
    fb = max(1, int(cfg.frames_per_block))
    stride = int(cfg.block_stride) if cfg.block_stride > 0 else hop * fb
    preroll = int(cfg.preroll) if cfg.preroll >= 0 else N
    return N, hop, fb, stride, preroll


def frame_starts(cfg, first_col, ncols):
    """First sample of each column's frame (frame_start_abs in jade_gpu.cu); negative: the frame reaches into the zeros
    that precede the stream."""
    _, hop, fb, stride, preroll = _geometry(cfg)
    j = np.arange(first_col, first_col + ncols, dtype=np.int64)
    return (j // fb) * stride + (j % fb) * hop - preroll


def channel_power(cfg, x, first_col, ncols, window=None):
    """x [channels][nsamples] float32 -> |X_c[k]|^2 * power_scale [ncols][channels][N/2+1], float64.  Samples outside
    [0, nsamples) are zeros (the pre-roll and the end of the stream)."""
    N = int(cfg.fft_size)
    w = (O.window(int(cfg.window), N) if window is None else np.asarray(window, np.float32)).astype(np.float64)
    x = np.asarray(x)
    ch, n = x.shape
    starts = frame_starts(cfg, first_col, ncols)
    out = np.empty((ncols, ch, N // 2 + 1), np.float64)
    step = max(1, (1 << 22) // (N * ch))
    for a in range(0, ncols, step):
        b = min(ncols, a + step)
        idx = starts[a:b, None] + np.arange(N)[None, :]
        ok = (idx >= 0) & (idx < n)
        fr = np.where(ok[:, None, :], x[:, np.clip(idx, 0, n - 1)].transpose(1, 0, 2).astype(np.float64), 0.0)
        X = np.fft.rfft(fr * w, axis=-1)
        out[a:b] = X.real ** 2 + X.imag ** 2
    return out * float(np.float32(cfg.power_scale) if cfg.power_scale > 0 else 1.0)


def mix(cfg, pc):
    """Channel mix of oracle/jade_oracle.cpp (and Spectrogram.cpp): pc [..., channels, bins] -> (p [..., bins], E [...])."""
    m = int(cfg.mix_mode)
    ch = pc.shape[-2]
    if m == MIX_ABSMEAN:
        p = pc.sum(axis=-2) / ch
        return p, p.sum(axis=-1)
    if m == MIX_MAX:
        p = np.maximum(pc.max(axis=-2), 0.0)
        src = pc
    elif m == MIX_MIN:
        p = np.minimum(pc.min(axis=-2), 1000000.0)  # the reference's start value: Min never exceeds 1e6
        src = pc
    else:
        c = 0 if m == MIX_LEFT or ch == 1 else 1
        p = pc[..., c, :]
        src = pc[..., c:c + 1, :]
    return p, src.sum(axis=-1).max(axis=-1)


def to_db(p):
    return 10.0 * np.log10(p + FLOOR)


def row_bins(cfg):
    """Per displayed row (top row first, as the pixels are stored): the bin range [lo, hi) it shows, None for one bin per
    row.  Returns (lo, hi, pooled)."""
    from jadespectrogram_b200 import _capi
    N = int(cfg.fft_size)
    B = N // 2 + 1
    rm = int(cfg.row_map)
    if rm == ROWS_LOG_MAXPOOL:
        R = int(cfg.rows)
        lo, hi = np.zeros(R, np.int32), np.zeros(R, np.int32)
        _capi.load().jade_log_rows(float(cfg.sample_rate), N, R, float(cfg.fmin), float(cfg.fmax), lo.ctypes.data, hi.ctypes.data)
    else:
        if rm == ROWS_LINEAR_CROP:
            a, b = C.c_int(), C.c_int()
            _capi.load().jade_linear_crop(float(cfg.sample_rate), B, float(cfg.fmin), float(cfg.fmax), C.byref(a), C.byref(b))
            k0, k1 = a.value, b.value
        else:
            k0, k1 = 0, B
        lo = np.arange(k0, k1, dtype=np.int32)
        hi = lo + 1
    if cfg.flip_y:
        lo, hi = lo[::-1], hi[::-1]
    return np.ascontiguousarray(lo), np.ascontiguousarray(hi), rm == ROWS_LOG_MAXPOOL


def rows_max(v, lo, hi, pooled):
    """v [..., bins] -> [..., rows]: the row map applied to a per-bin quantity (band maximum for pooled rows)."""
    if not pooled:
        return v[..., lo]
    return np.stack([v[..., a:b].max(axis=-1) for a, b in zip(lo, hi)], axis=-1)


class Ref:
    """The float64 reference of columns [first_col, first_col + ncols) of one stream x [channels][nsamples]."""

    def __init__(self, cfg, x, first_col, ncols, window=None, power=None):
        """power: channel_power() of the same columns, computed once for several configurations (power_scale 1)."""
        self.N = int(cfg.fft_size)
        if power is None:
            power = channel_power(cfg, x, first_col, ncols, window)
        elif cfg.power_scale > 0 and cfg.power_scale != 1.0:
            power = power * float(np.float32(cfg.power_scale))
        self.p, self.E = mix(cfg, power)
        self.db = to_db(self.p)
        self.lo, self.hi, self.pooled = row_bins(cfg)

    def tol(self):
        """(M64, allowed |M_gpu - M64| per bin, floor term per column)."""
        m = np.sqrt(self.p + FLOOR)
        floor = EPS32 * np.sqrt(np.log2(self.N) * self.E / self.N)[..., None]
        return m, A * floor + (B_REL + DB32) * m, floor

    def rows_db(self):
        return rows_max(self.db, self.lo, self.hi, self.pooled)

    def pixels(self, pal, pmin, pmax):
        """Reference ARGB pixels [ncols][rows]: the float32-rounded dB through the oracle palette's lookup."""
        pal.set_value_range(float(pmin), float(pmax))
        return pal.lookup(self.rows_db().astype(np.float32)).astype(np.uint32) | np.uint32(0xFF000000)


def db_errors(db_gpu, ref):
    """Normalised errors of dB values db_gpu [ncols][bins] against ref: dict(frac = worst |dM| / allowed, a = worst
    |dM| / (eps32 sqrt(log2 N E / N)) on bins more than 40 dB below their frame's peak, b = worst |dM| / M64 on the other bins where the floor term is
    the smaller one,
    ddb = worst |dB - dB64| on bins whose floor term is under a tenth of the relative term)."""
    assert db_gpu.shape == ref.p.shape, (db_gpu.shape, ref.p.shape)
    m, tol, floor = ref.tol()
    mg = np.sqrt(10.0 ** (db_gpu.astype(np.float64) / 10.0))
    d = np.abs(mg - m)
    loud = ref.db >= ref.db.max(axis=-1, keepdims=True) - 40.0
    clear = A * floor <= 0.1 * B_REL * m
    a = d / np.where(floor > 0, floor, np.inf)
    rel = loud & (A * floor <= B_REL * m)
    return dict(frac=float((d / tol).max()), a=float(a[~loud].max()) if (~loud).any() else 0.0,
                b=float((d / m)[rel].max()) if rel.any() else 0.0,
                ddb=float(np.abs(db_gpu.astype(np.float64) - ref.db)[clear].max()) if clear.any() else 0.0)


def check_db64(db_gpu, ref, label=""):
    """|M_gpu - M64| within the bound of the module docstring on every bin, and on bins whose floor term is negligible
    |dB - dB64| <= 20 log10(1 + 1.1 (B_REL + DB32)) (2.3e-4 dB).  Returns db_errors()."""
    e = db_errors(db_gpu, ref)
    assert e["frac"] <= 1.0, f"{label}: magnitude error {e['frac']:.2f}x the float64 bound (a {e['a']:.2f}, b {e['b']:.2e})"
    lim = 20.0 * np.log10(1.0 + 1.1 * (B_REL + DB32))
    assert e["ddb"] <= lim, f"{label}: dB differs from float64 by {e['ddb']:.2e} dB on bins well above the noise floor"
    return e


def check_pixels64(pix_gpu, ref, pal, pmin, pmax, ncolors, label=""):
    """Pixels [ncols][rows] against the reference's palette lookup; a pixel may differ only where the float64 dB of its
    row lies within the row's dB tolerance (check_db64's bound, for pooled rows the largest over the band) of a palette
    index edge or of the range ends -- parity.check_pixels' edge rule.  Returns the number of differing pixels."""
    want = ref.pixels(pal, pmin, pmax)
    assert pix_gpu.shape == want.shape, (pix_gpu.shape, want.shape)
    diff = pix_gpu != want
    if not diff.any():
        return 0
    lo_db, hi_db = min(pmin, pmax), max(pmin, pmax)
    m, tol, _ = ref.tol()
    tol_db = rows_max(20.0 * np.log10(1.0 + tol / m), ref.lo, ref.hi, ref.pooled) + 2e-5  # + the folded index FFMA's rounding
    v = ref.rows_db()
    mult = np.float32(ncolors) / (np.float32(hi_db) - np.float32(lo_db))
    pos = (np.clip(v, lo_db, hi_db) - lo_db) * float(mult)
    dist = np.abs(pos - np.round(pos)) / float(mult)
    near = (dist <= tol_db) | (np.abs(v - hi_db) <= tol_db) | (np.abs(v - lo_db) <= tol_db)
    bad = diff & ~near
    assert not bad.any(), f"{label}: {bad.sum()} of {diff.sum()} differing pixels are away from a palette edge"
    return int(diff.sum())


# ---- inputs that drive every level, bin, frame offset and stereo lane -------------------------------------------------

LEVELS = (1.0, 1e-3, 1e-5, 1e-6, 3e-7)


def _noise_sweep(rng, n, amp):
    t = np.arange(n) / n
    return (amp * (0.8 * np.sin(2 * np.pi * (0.01 * n * t + 0.2 * n * t * t)) + 0.2 * rng.uniform(-1, 1, n))).astype(np.float32)


def stream(kind, i, ch, n, N, hop, seed=1):
    """One stream [ch][n] float32 of a family of inputs (i: member of the family):
      level    noise + sweep at LEVELS[i % 5]; a stretch of exact zeros and one of subnormal samples in the middle, each
               long enough to hold whole silent frames
      bins     a comb of bin-centred cosines (period N, so every frame sees exactly these bins): bins k = i mod 8, DC and
               Nyquist included, at random phases
      impulse  unit impulses N + hop apart, so that each frame holds at most one; member i places them at frame offsets
               impulse_offsets(N, hop)[i::8] (|X_k|^2 = w[n0]^2 for every k)
      stereo   channel 1 derived from channel 0: silent, channel 0 silent, equal, opposite, 1e-6 times channel 0
      loud     noise + sweep at amplitude 1e3 and 3e4 (the upper palette clamp, u8 saturation, Min's 1e6 start)"""
    rng = np.random.default_rng(seed * 7919 + i * 31 + sum(map(ord, kind)))
    x = np.zeros((ch, n), np.float32)
    if kind == "level":
        amp = LEVELS[i % len(LEVELS)]
        for c in range(ch):
            x[c] = _noise_sweep(rng, n, amp * (1.0 - 0.1 * c))
        quiet = 2 * N + hop
        a = n // 4
        x[:, a:a + quiet] = 0.0
        sub = x[:, n // 2:n // 2 + quiet]
        sub[:] = rng.choice([-1.0, 1.0], sub.shape) * rng.uniform(1e-45, 1e-38, sub.shape)
    elif kind == "bins":
        spec = np.zeros(N // 2 + 1, np.complex128)
        ks = np.arange(i % 8, N // 2 + 1, 8)
        spec[ks] = np.exp(2j * np.pi * rng.random(ks.size))
        spec[0] = spec[0].real
        spec[-1] = spec[-1].real if ks[-1] == N // 2 else 0.0
        period = np.fft.irfft(spec, N)
        period *= 0.5 / np.abs(period).max()
        for c in range(ch):
            x[c] = np.tile(np.roll(period, 37 * c), n // N + 1)[:n]
    elif kind == "impulse":
        offs = impulse_offsets(N, hop)[i::8]
        D = N + hop
        for m, r in enumerate(offs):
            t = m * D + N + r
            if t < n:
                x[:, t] = 1.0
    elif kind == "stereo":
        base = _noise_sweep(rng, n, 0.5)
        x[:] = base
        if ch > 1:
            k = i % 5
            if k == 0:
                x[1] = 0.0
            elif k == 1:
                x[0] = 0.0
            elif k == 3:
                x[1] = -base
            elif k == 4:
                x[1] = base * np.float32(1e-6)
    elif kind == "loud":
        for c in range(ch):
            x[c] = _noise_sweep(rng, n, (1e3, 3e4)[i % 2])
    else:
        raise ValueError(kind)
    return x


def impulse_offsets(N, hop):
    """Sample positions (mod hop) of the impulses: every residue when hop <= 512 (each impulse is seen at ceil(N / hop)
    frame offsets r, r + hop, ..., so all N offsets are covered), else 64 residues spread over [0, hop)."""
    limit = 512 if hop <= 512 else 64
    if hop <= limit:
        return np.arange(hop)
    return np.unique(np.linspace(0, hop - 1, limit).round().astype(np.int64))


def stream_length(N, hop, offsets_per_stream):
    """Samples per stream: room for the level stretches and for `offsets_per_stream` impulses, a multiple of hop."""
    n = max(10 * (N + hop), (offsets_per_stream + 2) * (N + hop))
    return -(-n // hop) * hop


def batch(kinds, ch, N, hop, n, seed=1):
    """[(kind, i), ...] -> [streams][ch][n] float32."""
    return np.stack([stream(k, i, ch, n, N, hop, seed) for k, i in kinds])


def standard_kinds(ch, N, hop, extra_levels=0):
    """Every family once: 5 levels, 8 comb members, 8 impulse members, the stereo identities (two or more channels) and
    2 loud streams; extra_levels more level streams (long launches)."""
    kinds = [("level", i) for i in range(5)] + [("bins", i) for i in range(8)] + [("impulse", i) for i in range(8)]
    if ch > 1:
        kinds += [("stereo", i) for i in range(5)]
    kinds += [("loud", i) for i in range(2)] + [("level", 5 + i) for i in range(extra_levels)]
    return kinds
