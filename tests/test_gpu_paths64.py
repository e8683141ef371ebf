"""The paths into the kernels that tests/test_gpu_routes64.py does not take, against the float64 reference (tests/ref64.py).

test_gpu_routes64.py pins the arithmetic of every instantiation through one path: jade_render_device from column 0 over
whole, contiguous streams, the default pre-roll, one frame per block, palettes of 255 or 256 colours.  The rows here change
which samples a kernel reads, where it writes and which kernel runs, and compare every value with the same float64 bound
(ref64.check_db64 / ref64.check_pixels64) on the inputs of ref64.standard_kinds (fewer streams for N >= 16384):

  geometry       feed 10 % (ten frames per N-sample block: the division form of frame_start and odd hops) and 25 %, three
                 frames per block that are not evenly spaced, pre-roll 0, odd and 3 N + 2, hop 3 N / 2 (gaps between frames)
  channels       Left / Right on two and three channels for every kernel that takes a one-channel mix
  windows        first_col 1, mid-stream and near the end, windows running past the end of the stream, channel and stream
                 strides padded with NaN (a read outside [0, nsamples) turns a value into NaN), guard columns after the
                 output (a write past the launch's columns changes them), long-run launches starting after column 0, RGBA8
  palette        the palette lengths at which each configuration changes kernel (every kernel keeps the palette in shared
                 memory), one length either side; 1- and 2-colour tables; the restore of jade_set_palette when no kernel fits
  palette_cl     pkcl65536 with one channel, which no palette length reaches (see the row)
  streaming      jade_push_samples with seeded random push sizes on a ring of prime width: block emission at feed 10 %, a
                 paused stretch, jade_set_window between pushes, a push larger than the ring, polled pixel-only and dB
                 fetches, jade_recolor_ring / jade_read_ring_db after a palette and range change
  stream_run     one push long enough for the long-run (tensor-memory ring) instantiations while streaming
  chunks         jade_render_batch split into many column and stream chunks, pageable and jade_host_alloc buffers

Each group runs in a child process with JADE_TRACE_LAUNCH=1 (one `[jade] <kernel>[+run][+db][+u8] grid ...` line per
launch; the switch is read once per process) and without the experiment switches, except where GROUP_ENV names one and
the group's rows say why.  The test asserts that each row launched the instantiations it names and prints, per row, the
share of the float64 bound used and the number of pixels that differ from the reference (only allowed at palette edges).
"""
import bisect
import json
import os
import pathlib
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest

ROOT = pathlib.Path(__file__).resolve().parent.parent

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

JADE = ("jade", 256, -50.0, 50.0)
SWITCHES = ("JADE_PK_LOAD", "JADE_RUN_MIN", "JADE_N16384", "JADE_N65536", "JADE_MAX_GRID", "JADE_BLOCKS_PER_SM",
            "JADE_CHUNK_MB", "JADE_PIPE_DEPTH")
GROUP_ENV = {
    "palette_cl": {"JADE_N65536": "cl"},  # the only route to pkcl65536 with one contributing channel (row docstring)
    "stream_run": {"JADE_RUN_MIN": "2"},  # keeps the pinned staging of the long push near 100 MB (row docstring)
    "chunks": {"JADE_CHUNK_MB": "1"},     # many chunks from test-sized inputs (read once per process)
}
SENT_PIX = 0x5A5A5A5A                     # guard columns: alpha 0x5A, never a baked pixel (alpha 0xFF)
SENT_DB = np.float32(-7777.0)

# kernel family -> base configuration (hop N / 4 unless a row says otherwise)
FAM = {
    "pksmall<2>": dict(fft_size=128, channels=1),
    "pksmall<4>": dict(fft_size=256, channels=2),
    "pksmall<8>": dict(fft_size=512, channels=1),
    "pksmall<16>": dict(fft_size=1024, channels=2),
    "pk2048": dict(fft_size=2048, channels=1),
    "pkz2048": dict(fft_size=2048, channels=2),
    "pk3<16384>": dict(fft_size=16384, channels=1),
    "pkcta<2>": dict(fft_size=4096, channels=1),
    "pkcta<4>": dict(fft_size=8192, channels=2),
    "pkcta<8>": dict(fft_size=16384, channels=2),
    "pkcta<16>": dict(fft_size=32768, channels=1),
    "pkcl3<65536>": dict(fft_size=65536, channels=1),
    "pkcl65536": dict(fft_size=65536, channels=2),
    "warp<8>": dict(fft_size=512, channels=1, flip_y=0),
    "cta<4>": dict(fft_size=8192, channels=1, db_precise=1),
}


def _expect(fam, guard=True):
    """Instantiations a dB-storing and a pixel-only launch (256-colour jade palette) of a family must show; `guard`: the
    row also has launches whose frames are not 8-byte aligned."""
    if fam.startswith(("pkcl", "warp", "cta")):
        return [fam]
    if fam.startswith("pkcta"):
        return [fam + "+db", fam]
    pix = fam + "+u8" if fam in ("pkz2048", "pk3<16384>") else fam
    return [fam + "+db", pix] + ([fam + "-guard"] if guard else [])


def _row(name, group, kind, cfg, expect, **kw):
    return dict(name=name, group=group, kind=kind, cfg=cfg, expect=expect, **kw)


GEOMS = [("feed10", lambda N: dict(feed_percent=10)), ("feed25", lambda N: dict(feed_percent=25)),
         ("fb3", lambda N: dict(hop=N // 4, frames_per_block=3, block_stride=N)),
         ("preroll0", lambda N: dict(hop=N // 4, preroll=0)), ("preroll_odd", lambda N: dict(hop=N // 4, preroll=N // 2 + 3)),
         ("preroll3N+2", lambda N: dict(hop=N // 4, preroll=3 * N + 2)), ("hop3N/2", lambda N: dict(hop=3 * N // 2))]


def _rows():
    R = []
    # geometry: every family, every geometry, dB-storing and pixel-only
    for fam, cfg in FAM.items():
        exp = _expect(fam) + (["pk2048-ldg+db"] if fam == "pk2048" else [])  # pre-roll 3N+2: 8- but not 16-byte aligned
        R.append(_row(f"geometry {fam}", "geometry", "geometry", cfg, exp))
    # channels: Left / Right on two and three channels, every kernel with a one-channel mix
    one = [("pksmall<4>", dict(fft_size=256)), ("pksmall<16>", dict(fft_size=1024)), ("pk2048", dict(fft_size=2048)),
           ("pk3<16384>", dict(fft_size=16384)), ("pkcta<2>", dict(fft_size=4096)), ("pkcta<16>", dict(fft_size=32768)),
           ("pkcl3<65536>", dict(fft_size=65536)), ("warp<8>", dict(fft_size=512, flip_y=0)),
           ("cta<2>", dict(fft_size=4096, flip_y=0))]
    for fam, cfg in one:
        for mix in ("left", "right"):
            for ch in (2, 3):
                R.append(_row(f"{fam} {mix} ch{ch}", "channels", "render", dict(cfg, channels=ch, mix_mode=mix), _expect(fam),
                              launches=[(True, 0), (False, 0), (True, 1)]))
    R.append(_row("pk2048+run right ch2", "channels", "render", dict(fft_size=2048, hop=512, channels=2, mix_mode="right"),
                  ["pk2048+run+db", "pk2048+run"], launches=[(True, 0), (False, 0)], min_frames=44000))
    # windows and strides
    for fam in ("pksmall<4>", "pksmall<8>", "pk2048", "pkz2048", "pk3<16384>", "pkcta<4>", "pkcta<16>", "pkcl3<65536>",
                "pkcl65536", "warp<8>", "cta<4>"):
        R.append(_row(f"windows {fam}", "windows", "windows", FAM[fam], _expect(fam)))
    for hop in (256, 512):
        R.append(_row(f"pk2048+run window hop{hop}", "windows", "render", dict(fft_size=2048, hop=hop, channels=1),
                      ["pk2048+run+db", "pk2048+run"], launches=[(True, 0), (False, 0)], min_frames=44000, first=7, tail=2))
    R.append(_row("pkz2048+run window", "windows", "render", dict(fft_size=2048, hop=512, channels=2),
                  ["pkz2048+run+db", "pkz2048+run+u8"], launches=[(True, 0), (False, 0)], min_frames=34000, first=5, tail=3))
    # palette routes: (configuration, the routes from 256 colours up, instantiations the renders must show).  A packed
    # N <= 2048 kernel falls back to the general warp kernel where that one holds more colours (one channel at N = 512,
    # 1024, 2048); a two-channel sum holds more in the packed kernel, so it goes straight to the refusal.  The general cta
    # kernels hold fewer colours than every packed N >= 4096 kernel, so no palette length routes to them: their row checks
    # their own limit and the refusal.
    pal = [
        ("pksmall<2> mono", dict(fft_size=128, channels=1), ["pksmall<2>", "ERR"], ["pksmall<2>+db", "pksmall<2>"]),
        ("pksmall<8> mono", dict(fft_size=512, channels=1), ["pksmall<8>", "warp<8>", "ERR"], ["pksmall<8>+db", "warp<8>"]),
        ("pksmall<16> mono", dict(fft_size=1024, channels=1), ["pksmall<16>", "warp<16>", "ERR"], ["pksmall<16>+db", "warp<16>"]),
        ("pksmall<16> stereo", dict(fft_size=1024, channels=2), ["pksmall<16>", "ERR"], ["pksmall<16>+db"]),
        ("pk2048 mono", dict(fft_size=2048, channels=1), ["pk2048", "warp<32>", "ERR"], ["pk2048+db", "warp<32>"]),
        ("pk2048 stereo", dict(fft_size=2048, channels=2), ["pkz2048", "pk2048", "ERR"],
         ["pkz2048+db", "pk2048+db", "pk2048", "pk2048-ldg+db", "pk2048-ldg", "pk2048-guard"]),
        ("pk3<16384> mono", dict(fft_size=16384, channels=1), ["pk3<16384>", "pkcta<8>", "ERR"], ["pk3<16384>+db", "pkcta<8>+db", "pkcta<8>"]),
        ("pkcta<2> stereo", dict(fft_size=4096, channels=2), ["pkcta<2>", "ERR"], ["pkcta<2>+db"]),
        ("pkcta<16> mono", dict(fft_size=32768, channels=1), ["pkcta<16>", "ERR"], ["pkcta<16>+db"]),
        ("pkcl3<65536> mono", dict(fft_size=65536, channels=1), ["pkcl3<65536>", "ERR"], ["pkcl3<65536>"]),
        ("pkcl65536 stereo", dict(fft_size=65536, channels=2), ["pkcl65536", "ERR"], ["pkcl65536"]),
        ("warp<4> precise", dict(fft_size=256, channels=1, db_precise=1), ["warp<4>", "ERR"], ["warp<4>"]),
        ("cta<4> unflipped", dict(fft_size=8192, channels=1, flip_y=0), ["cta<4>", "ERR"], ["cta<4>"]),
    ]
    for name, cfg, routes, exp in pal:
        R.append(_row(f"palette {name}", "palette", "palette", dict(cfg, hop=cfg["fft_size"] // 4), exp, routes=routes))
    # pkcl65536 with one channel: its table limit lies below pkcl3's, so no palette length routes a one-channel mix to it
    # (the palette rows show pkcl3<65536> -> ERR); the JADE_N65536=cl switch is the only way to launch it
    for ch, mix in ((1, "absmean"), (2, "right")):
        R.append(_row(f"pkcl65536 one channel ch{ch} {mix}", "palette_cl", "render",
                      dict(fft_size=65536, hop=16384, channels=ch, mix_mode=mix), ["pkcl65536"], launches=[(True, 0), (False, 0)]))
    # streaming: one configuration per family
    st = [
        ("pksmall<8> feed10 block", dict(fft_size=512, channels=1, feed_percent=10), ["pksmall<8>-guard"]),
        ("pksmall<4> stereo", dict(fft_size=256, hop=64, channels=2), ["pksmall<4>+db"]),
        ("pk2048 mono", dict(fft_size=2048, hop=512, channels=1), ["pk2048+db"]),
        ("pk2048 right feed25 block", dict(fft_size=2048, channels=2, mix_mode="right", feed_percent=25), ["pk2048+db"]),
        ("pkz2048 feed10 block", dict(fft_size=2048, channels=2, feed_percent=10), ["pkz2048-guard"]),
        ("pkz2048 stereo", dict(fft_size=2048, hop=512, channels=2), ["pkz2048+db"]),
        ("pk3<16384>", dict(fft_size=16384, hop=4096, channels=1), ["pk3<16384>+db"]),
        ("pkcta<4> stereo", dict(fft_size=8192, hop=2048, channels=2), ["pkcta<4>+db"]),
        ("pkcta<8> stereo", dict(fft_size=16384, hop=4096, channels=2), ["pkcta<8>+db"]),
        ("pkcta<16> mono", dict(fft_size=32768, hop=8192, channels=1), ["pkcta<16>+db"]),
        ("pkcl3<65536>", dict(fft_size=65536, hop=16384, channels=1), ["pkcl3<65536>"]),
        ("pkcl65536", dict(fft_size=65536, hop=16384, channels=2), ["pkcl65536"]),
        ("warp<16> crop", dict(fft_size=1024, hop=256, channels=1, row_map="linear_crop", fmin=1000.0, fmax=8000.0), ["warp<16>"]),
        ("cta<2> log rows", dict(fft_size=4096, hop=1024, channels=1, row_map="log_maxpool", rows=64, fmin=50.0, fmax=20000.0), ["cta<2>"]),
        ("warp<8> unflipped max", dict(fft_size=512, hop=128, channels=2, mix_mode="max", flip_y=0), ["warp<8>"]),
        ("cta<4> precise min", dict(fft_size=8192, hop=2048, channels=2, mix_mode="min", db_precise=1), ["cta<4>"]),
    ]
    for k, (name, cfg, exp) in enumerate(st):
        R.append(_row(f"stream {name}", "streaming", "stream", cfg, exp, seed=100 + k))
    R.append(_row("stream pk2048+run mono hop256", "stream_run", "stream_run", dict(fft_size=2048, hop=256, channels=1),
                  ["pk2048+run+db"]))
    R.append(_row("stream pkz2048+run stereo hop512", "stream_run", "stream_run", dict(fft_size=2048, hop=512, channels=2),
                  ["pkz2048+run+db"]))
    # host chunks: (configuration, streams, first column, columns or None = to the end less 2, pinned, dB)
    ch = [
        ("pkz2048 pageable db", dict(fft_size=2048, hop=512, channels=2), 6, 5, None, False, True, ["pkz2048+db"]),
        ("pkz2048 pinned db", dict(fft_size=2048, hop=512, channels=2), 6, 5, None, True, True, ["pkz2048+db"]),
        ("pkz2048 pageable pixels, stream chunks", dict(fft_size=2048, hop=512, channels=2), 13, 9, 40, False, False, ["pkz2048+u8"]),
        ("pkz2048 pinned pixels, stream chunks", dict(fft_size=2048, hop=512, channels=2), 13, 9, 40, True, False, ["pkz2048+u8"]),
        ("pksmall<16> feed10 pinned db", dict(fft_size=1024, channels=1, feed_percent=10), 5, 11, None, True, True, ["pksmall<16>-guard"]),
        ("pk2048 right pageable db", dict(fft_size=2048, hop=512, channels=2, mix_mode="right"), 4, 3, None, False, True, ["pk2048+db"]),
        ("pk3<16384> pinned db", dict(fft_size=16384, hop=4096, channels=1), 4, 2, None, True, True, ["pk3<16384>+db"]),
        ("cta<2> log rows pageable db", dict(fft_size=4096, hop=1024, channels=1, row_map="log_maxpool", rows=64, fmin=50.0,
                                              fmax=20000.0), 4, 3, None, False, True, ["cta<2>"]),
    ]
    for name, cfg, S, first, ncols, pinned, want_db, exp in ch:
        R.append(_row(f"chunks {name}", "chunks", "chunks", cfg, exp, streams=S, first=first, ncols=ncols, pinned=pinned,
                      want_db=want_db))
    return R


ROWS = _rows()
GROUPS = sorted({r["group"] for r in ROWS})


# ---- child process: helpers ------------------------------------------------------------------------------------------

def _kinds(ch, N, hop):
    import ref64
    if N < 16384:
        return ref64.standard_kinds(ch, N, hop)
    k = [("level", 0), ("level", 3), ("level", 4), ("bins", 0), ("bins", 5), ("impulse", 0), ("impulse", 5), ("loud", 1)]
    return k + ([("stereo", 0), ("stereo", 3)] if ch > 1 else [])


def _engine(cfg, **over):
    from jadespectrogram_b200 import Engine
    kw = dict(sample_rate=48000.0, window="hann", mix_mode="absmean")
    kw.update(cfg)
    kw.update(over)
    return Engine(0, **kw)


def _inputs(eng, min_frames=0):
    """Streams of ref64.standard_kinds (fewer for N >= 16384) for the engine's geometry; enough extra level streams for
    `min_frames` columns in all."""
    import ref64
    c = eng.get_config()
    N, ch = c.fft_size, c.channels
    hop = max(1, c.block_stride // c.frames_per_block)
    kinds = _kinds(ch, N, hop)
    n = ref64.stream_length(N, hop, -(-len(ref64.impulse_offsets(N, hop)) // 8))
    if min_frames:
        cols = eng.columns_for(n)
        kinds = kinds + [("level", 5 + i) for i in range(max(0, -(-min_frames // cols) - len(kinds)))]
    return ref64.batch(kinds, ch, N, hop, n), kinds


def _powers(eng, x, first, ncols, window=None):
    import ref64
    c1 = eng.get_config()
    c1.power_scale = 1.0
    return [ref64.channel_power(c1, x[s], first, ncols, window) for s in range(x.shape[0])]


def _refs(eng, powers, a=0, b=None):
    import ref64
    cfg = eng.get_config()
    return [ref64.Ref(cfg, None, 0, 0, power=p[a:b]) for p in powers]


def _argb(pix):
    """RGBA8 pixels (bytes R, G, B, A) -> the ARGB32 words of the reference."""
    p = pix.astype(np.uint32)
    return (p & np.uint32(0xFF00FF00)) | ((p >> np.uint32(16)) & np.uint32(0xFF)) | ((p & np.uint32(0xFF)) << np.uint32(16))


def _check(rec, label, refs, pix, db, pal=JADE):
    import oracle_lib as O
    import ref64
    scheme, npal, pmin, pmax = pal
    opal = O.Palette(npal, O.PAL[scheme])
    worst = dict(frac=0.0, a=0.0, b=0.0, ddb=0.0)
    nd = 0
    for s, r in enumerate(refs):
        lab = f"{rec['row']}: {label} stream {s}"
        if db is not None:
            e = ref64.check_db64(db[s], r, lab)
            worst = {k: max(worst[k], e[k]) for k in worst}
        nd += ref64.check_pixels64(pix[s], r, opal, pmin, pmax, npal, lab)
    rec["launches"].append(dict(label=label, pixels_differing=nd, **worst))


def _render(eng, x, first, ncols, want_db, off=0, pads=(0, 0), guard=3):
    """render_device over x [streams][ch][n] laid out with `pads` = (+floats per channel, +floats per stream) of NaN
    between them, 16 NaN floats in front, `off` floats of misalignment, and `guard` sentinel columns after the output."""
    import torch
    S, ch, n = x.shape
    cs = n + pads[0]
    ss = ch * cs + pads[1]
    base = 16 + off
    host = np.full(base + S * ss + 16, np.nan, np.float32)
    v = host[base:base + S * ss].reshape(S, ss)
    for c in range(ch):
        v[:, c * cs:c * cs + n] = x[:, c]
    R, B = eng.R, eng.B
    d_in = torch.from_numpy(host).cuda()
    d_pix = torch.full(((S * ncols + guard) * R,), SENT_PIX, dtype=torch.int32, device="cuda")
    d_db = torch.full(((S * ncols + guard) * B,), float(SENT_DB), dtype=torch.float32, device="cuda") if want_db else None
    torch.cuda.synchronize()  # the engine's stream does not wait for torch's
    eng.render_device(d_in.data_ptr() + 4 * base, S, n, ss, cs, first, ncols, d_pix.data_ptr(),
                      d_db.data_ptr() if want_db else None)
    eng.sync()
    pix = d_pix.cpu().numpy().view(np.uint32)
    assert (pix[S * ncols * R:] == SENT_PIX).all(), "pixels written after the last column of the last stream"
    db = None
    if want_db:
        d = d_db.cpu().numpy()
        assert (d[S * ncols * B:] == SENT_DB).all(), "dB values written after the last column of the last stream"
        db = d[:S * ncols * B].reshape(S, ncols, B)
    return pix[:S * ncols * R].reshape(S, ncols, R), db


def _set_pal(eng, pal):
    eng.set_palette_scheme(pal[0], pal[1])
    eng.set_value_range(pal[2], pal[3])


# ---- child process: row kinds -----------------------------------------------------------------------------------------

def _do_geometry(row, rec):
    N = row["cfg"]["fft_size"]
    for gname, g in GEOMS:
        eng = _engine(row["cfg"], **g(N))
        x, _ = _inputs(eng)
        total = eng.columns_for(x.shape[2])
        refs = _refs(eng, _powers(eng, x, 0, total))
        for want_db in (True, False):
            pix, db = _render(eng, x, 0, total, want_db)
            _check(rec, f"{gname} db={want_db}", refs, pix, db)
        eng.close()


def _do_render(row, rec):
    eng = _engine(row["cfg"])
    x, _ = _inputs(eng, row.get("min_frames", 0))
    total = eng.columns_for(x.shape[2])
    first = row.get("first", 0)
    ncols = total - first - row.get("tail", 0)
    refs = _refs(eng, _powers(eng, x, first, ncols))
    for want_db, off in row["launches"]:
        pix, db = _render(eng, x, first, ncols, want_db, off=off)
        _check(rec, f"cols [{first},{first + ncols}) db={want_db} off={off}", refs, pix, db)
    eng.close()


def _do_windows(row, rec):
    eng = _engine(row["cfg"])
    x, _ = _inputs(eng)
    total = eng.columns_for(x.shape[2])
    powers = _powers(eng, x, 0, total + 4)  # the columns after the end: frames of zeros (and the stream's tail)
    wins = [(1, total - 1), (total // 2, max(1, total // 4)), (total - 3, 3), (total - 4, 6), (total // 3, total - total // 3 + 3)]
    launches = [(a, n, True, (0, 0), 0) for a, n in wins] + [(1, total - 1, False, (0, 0), 0)]
    launches += [(0, total, True, p, 0) for p in ((1, 2), (2, 4), (4, 1))] + [(3, total - 2, False, (4, 4), 0)]
    for a, n, want_db, pads, off in launches:
        pix, db = _render(eng, x, a, n, want_db, off=off, pads=pads)
        _check(rec, f"cols [{a},{a + n}) db={want_db} pads={pads}", _refs(eng, powers, a, a + n), pix, db)
    eng.close()
    eng = _engine(row["cfg"], pixel_format="rgba8")
    for want_db in (False, True):
        pix, db = _render(eng, x, 0, total, want_db)
        _check(rec, f"rgba8 db={want_db}", _refs(eng, powers, 0, total), _argb(pix), db)
    eng.close()


def _route(eng, n):
    rc = eng.lib.jade_set_palette_scheme(eng.h, 6, int(n), 0)  # JADE_PAL_JADE
    return eng.kernel_name if rc == 0 else f"ERR{rc}"


def _route_changes(eng, lo=256, hi=65536):
    """[(first length of a route, route)] from `lo` colours up to `hi`: bisection (the shared memory a kernel needs grows
    with the table, so each route holds over one interval of lengths)."""
    out = [(lo, _route(eng, lo))]
    while not out[-1][1].startswith("ERR") and _route(eng, hi) != out[-1][1]:
        a, b, cur = out[-1][0], hi, out[-1][1]
        while b - a > 1:
            m = (a + b) // 2
            if _route(eng, m) == cur:
                a = m
            else:
                b = m
        out.append((b, _route(eng, b)))
    return out


def _do_palette(row, rec):
    from jadespectrogram_b200._capi import JADE_ERR_ARG
    eng = _engine(row["cfg"])
    x, _ = _inputs(eng)
    total = eng.columns_for(x.shape[2])
    refs = _refs(eng, _powers(eng, x, 0, total))
    changes = _route_changes(eng)
    rec["info"] = "routes " + ", ".join(f"{r} from {n}" for n, r in changes)
    assert [r if not r.startswith("ERR") else "ERR" for _, r in changes] == row["routes"], rec["info"]
    assert changes[-1][1] == f"ERR{JADE_ERR_ARG}", rec["info"]
    full = [(True, 0), (False, 0), (True, 1), (True, 2), (False, 2)]
    for k in range(1, len(changes)):
        c, route = changes[k]
        below = ("jade", c - 1, -50.0, 50.0)
        _set_pal(eng, below)
        assert eng.kernel_name == changes[k - 1][1]
        for want_db, off in [(True, 0), (False, 0)]:
            pix, db = _render(eng, x, 0, total, want_db, off=off)
            _check(rec, f"{c - 1} colours ({changes[k - 1][1]}) db={want_db} off={off}", refs, pix, db, below)
        if not route.startswith("ERR"):
            at = ("jade", c, -50.0, 50.0)
            _set_pal(eng, at)
            assert eng.kernel_name == route
            for want_db, off in (full if route == "pk2048" else [(True, 0), (False, 0)]):
                pix, db = _render(eng, x, 0, total, want_db, off=off)
                _check(rec, f"{c} colours ({route}) db={want_db} off={off}", refs, pix, db, at)
            continue
        # no kernel fits `c` colours: jade_set_palette fails with JADE_ERR_ARG and keeps the table, range and kernel
        pix0, _ = _render(eng, x, 0, total, False)
        probe = np.linspace(-60.0, 60.0, 4001, dtype=np.float32)
        lut0 = [eng.lookup_color(v) for v in probe]
        range0, name0 = eng.get_value_range(), eng.kernel_name
        rc = eng.lib.jade_set_palette_scheme(eng.h, 6, c, 0)
        assert rc == JADE_ERR_ARG, f"{c} colours: jade_set_palette returned {rc}, want JADE_ERR_ARG"
        assert eng.get_value_range() == range0, (eng.get_value_range(), range0)
        assert [eng.lookup_color(v) for v in probe] == lut0, "the previous table was not kept"
        assert eng.kernel_name == name0
        pix1, _ = _render(eng, x, 0, total, False)
        assert np.array_equal(pix1, pix0), "rendering changed after a refused palette"
        _check(rec, f"{c} colours refused, {c - 1} kept", refs, pix1, None, below)
    # one- and two-colour tables on the configuration's first route
    for npal in (1, 2):
        p = ("jade", npal, -50.0, 50.0)
        _set_pal(eng, p)
        assert eng.kernel_name == changes[0][1]
        pix, db = _render(eng, x, 0, total, True)
        _check(rec, f"{npal} colours", refs, pix, db, p)
    eng.close()


def _is_prime(n):
    return n > 1 and all(n % d for d in range(2, int(n ** 0.5) + 1))


class _Stream:
    """Drives one streaming engine and keeps, for every emitted column, the frame and window it shows."""

    def __init__(self, eng, x):
        self.eng, self.x = eng, x
        self.pos = 0
        self.window = "hann"
        self.ranges = []  # (first emitted index, end, frame - emitted index, window) per push
        self.got = {}     # emitted index -> (pixels, dB or None)
        self.k = 0

    def push(self, m):
        eng = self.eng
        e0 = eng.ring_info()[3]
        eng.push(self.x[:, self.pos:self.pos + m])
        self.pos += m
        e1 = eng.ring_info()[3]
        frames = eng.columns_for(self.pos)
        if e1 > e0:
            self.ranges.append((e0, e1, frames - e1, self.window))
        return frames

    def fetch(self, want_db=None):
        if want_db is None:
            want_db = self.k % 2 == 1  # alternate the polled pixel-only path and the dB path
            self.k += 1
        pix, db, first = self.eng.fetch(max_cols=self.eng.W, want_db=want_db)
        for i in range(len(pix)):
            self.got[first + i] = (pix[i], db[i] if want_db else None)

    def where(self, k):
        i = bisect.bisect_right([r[0] for r in self.ranges], k) - 1
        a, b, off, w = self.ranges[i]
        assert a <= k < b, (k, self.ranges[i])
        return k + off, w

    def runs(self, ks):
        """Emitted indices -> runs [(frame0, window, [indices])] of consecutive frames with one window."""
        out = []
        for k in sorted(ks):
            j, w = self.where(k)
            if out and out[-1][1] == w and out[-1][0] + len(out[-1][2]) == j:
                out[-1][2].append(k)
            else:
                out.append((j, w, [k]))
        return out


def _stream_check(st, rec, label, cols, pal=JADE):
    """cols: emitted index -> (pixels, dB or None); checked per run of frames against ref64 with that run's window."""
    import oracle_lib as O
    import ref64
    eng = st.eng
    cfg = eng.get_config()
    cfg.power_scale = 1.0
    N = cfg.fft_size
    for j0, w, ks in st.runs(cols):
        pw = ref64.channel_power(cfg, st.x, j0, len(ks), O.window(w, N))
        lab = f"{label} frames [{j0},{j0 + len(ks)}) {w}"
        _check(rec, lab, [ref64.Ref(cfg, None, 0, 0, power=pw)], np.stack([cols[k][0] for k in ks])[None], None, pal)
        sub = [i for i, k in enumerate(ks) if cols[k][1] is not None]
        if sub:
            _check(rec, lab + " dB", [ref64.Ref(cfg, None, 0, 0, power=pw[sub])], np.stack([cols[ks[i]][0] for i in sub])[None],
                   np.stack([cols[ks[i]][1] for i in sub])[None], pal)


def _do_stream(row, rec):
    import ref64
    cfg = row["cfg"]
    N = cfg["fft_size"]
    W = 73 if N <= 16384 else 37  # prime; >= 72 arms the polled fetch path (jade_push_samples)
    probe = _engine(cfg)
    c = probe.get_config()
    probe.close()
    hop_eff = c.block_stride / c.frames_per_block
    big = int(-(-(W + 8) * c.block_stride // c.frames_per_block)) + 2 * N  # more than a ring of columns in one push
    eng = _engine(cfg, ring_columns=W, max_push=big)
    rng = np.random.default_rng(row["seed"])
    n_total = int((2 * W + 120) * hop_eff) + big + 4 * N
    x = ref64.stream("level", 0, c.channels, n_total, N, int(hop_eff))
    st = _Stream(eng, x)
    small = max(1, int(3 * hop_eff))

    def until(frames):
        while eng.columns_for(st.pos) < frames:
            st.push(int(rng.integers(1, small + 1)))
            st.fetch()

    until(W + 10)                          # the ring has wrapped
    eng.set_window("blackmanharris")
    st.window = "blackmanharris"
    until(eng.columns_for(st.pos) + 15)
    eng.set_pause(True)                    # frames pass, nothing is emitted
    f0 = eng.columns_for(st.pos)
    until(f0 + 6)
    eng.set_pause(False)
    e0 = eng.ring_info()[3]
    f0 = st.push(big)                      # more than a ring: the oldest columns of the push are skipped
    assert eng.ring_info()[3] - e0 > W, "the long push did not overflow the ring"
    st.fetch(want_db=True)
    until(f0 + 12)
    eng.set_window("hann")
    st.window = "hann"
    until(eng.columns_for(st.pos) + 10)
    st.fetch(want_db=True)
    assert st.pos <= n_total
    _stream_check(st, rec, "fetched", st.got)
    # a palette and range change, then the whole ring re-coloured and read back
    pal = ("viridis", 256, -90.0, 10.0)
    _set_pal(eng, pal)
    ring_pix, ring_db = eng.recolor_ring(), eng.read_ring_db()
    em = eng.ring_info()[3]
    ring = {}
    for s in range(W):
        k = em - 1 - ((em - 1 - s) % W)
        ring[k] = (ring_pix[s], ring_db[s])
    _stream_check(st, rec, "ring", ring, pal)
    rec["info"] = f"ring {W}, {len(st.got)} columns fetched, {em} emitted, {eng.columns_for(st.pos)} frames"
    eng.close()


def _traced(fn):
    """Runs fn() with this process's stderr captured; returns the text (also passed on to stderr)."""
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile("w+") as f:
        os.dup2(f.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
        f.seek(0)
        text = f.read()
    sys.stderr.write(text)
    sys.stderr.flush()
    return text


RUN_LINE = re.compile(r"^\[jade\] (\S+) grid (\d+) x \d+ threads, smem \d+, blocks/SM (\d+), frames (\d+), units/block (\d+)")


def _do_stream_run(row, rec):
    """One push long enough for the long-run instantiation while streaming.  A launch takes the long-run form when it has
    at least JADE_RUN_MIN x grid x units-per-block frames; the grid and units are read from the trace of a long probe
    launch.  JADE_RUN_MIN is 2 in this group (16 by default): the push then needs ~3600 stereo frames of 512 samples, not
    ~28000, and its pinned staging (8 slots x max_push x channels x 4 B) stays near 100 MB instead of ~1 GB; with 2 every
    warp still walks several contiguous columns, so the ring-slot arithmetic between them runs."""
    import torch

    import ref64
    cfg = row["cfg"]
    N, hop, ch = cfg["fft_size"], cfg["hop"], cfg["channels"]
    run_min = int(os.environ["JADE_RUN_MIN"])
    eng = _engine(cfg)
    S, n = 100, 400 * hop
    d_in = torch.zeros(S * ch * n, dtype=torch.float32, device="cuda")
    ncols = eng.columns_for(n)
    d_pix = torch.empty(S * ncols * eng.R, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    print(f"[row] {row['name']}/probe", file=sys.stderr, flush=True)
    text = _traced(lambda: (eng.render_device(d_in.data_ptr(), S, n, ch * n, n, 0, ncols, d_pix.data_ptr()), eng.sync()))
    del d_in, d_pix
    eng.close()
    m = max((RUN_LINE.match(l) for l in text.splitlines() if RUN_LINE.match(l)), key=lambda m: int(m.group(4)))
    grid, bps, units = int(m.group(2)), int(m.group(3)), int(m.group(5))
    threshold = run_min * grid * units
    print(f"[row] {row['name']}", file=sys.stderr, flush=True)
    nbig = threshold + 5
    W = nbig
    while not _is_prime(W):
        W += 1
    eng = _engine(cfg, ring_columns=W, max_push=nbig * hop)
    x = ref64.stream("level", 0, ch, (W + 200) * hop + nbig * hop + 2 * N, N, hop)
    st = _Stream(eng, x)
    while eng.ring_info()[3] < W - nbig + 10:  # so that the long push wraps around the end of the ring
        st.push(3 * hop)
        st.fetch()
    e0 = eng.ring_info()[3]
    st.push(nbig * hop)
    assert eng.ring_info()[3] - e0 == nbig and (e0 % W) + nbig > W, (e0, nbig, W)
    st.fetch(want_db=True)
    for _ in range(3):
        st.push(2 * hop)
        st.fetch(want_db=False)
    _stream_check(st, rec, "fetched", st.got)
    rec["info"] = (f"probe grid {grid} (blocks/SM {bps}) x {units} units -> long runs from {threshold} frames; "
                   f"push of {nbig} columns into a ring of {W} from slot {e0 % W}")
    eng.close()


def _do_chunks(row, rec):
    from jadespectrogram_b200.engine import host_alloc, host_free
    eng = _engine(row["cfg"])
    x, _ = _inputs(eng)
    x = x[:row["streams"]]
    S, ch, n = x.shape
    total = eng.columns_for(n)
    first = row["first"]
    ncols = row["ncols"] or total - first - 2
    bufs = []
    if row["pinned"]:
        xs = host_alloc(x.shape, np.float32)
        xs[:] = x
        pix = host_alloc((S, ncols, eng.R), np.uint32)
        db = host_alloc((S, ncols, eng.B), np.float32) if row["want_db"] else None
        bufs = [b for b in (xs, pix, db) if b is not None]
    else:
        xs = x
        pix = np.empty((S, ncols, eng.R), np.uint32)
        db = np.empty((S, ncols, eng.B), np.float32) if row["want_db"] else None
    eng.render_batch(xs, first_col=first, ncols=ncols, out_pix=pix, out_db=db)
    pix, db = pix.copy(), (db.copy() if db is not None else None)
    for b in bufs:
        host_free(b)
    col_bytes = eng.R * 4 + (eng.B * 4 if row["want_db"] else 0)
    rec["info"] = f"{S} streams x columns [{first},{first + ncols}), {col_bytes * ncols * S / 2 ** 20:.1f} MB of output in 1 MB chunks"
    _check(rec, "render_batch", _refs(eng, _powers(eng, x, first, ncols)), pix, db)
    eng.close()


def _run_group(group, outdir):
    sys.path.insert(0, str(ROOT))
    sys.path.insert(0, str(ROOT / "tests"))
    kinds = dict(geometry=_do_geometry, render=_do_render, windows=_do_windows, palette=_do_palette, stream=_do_stream,
                 stream_run=_do_stream_run, chunks=_do_chunks)
    results = []
    for row in [r for r in ROWS if r["group"] == group]:
        print(f"[row] {row['name']}", file=sys.stderr, flush=True)
        rec = dict(row=row["name"], launches=[], error=None, info="")
        results.append(rec)
        try:
            kinds[row["kind"]](row, rec)
        except Exception as ex:  # noqa: BLE001 -- reported to the parent, which fails the test
            import traceback
            traceback.print_exc()
            rec["error"] = f"{type(ex).__name__}: {ex}"
    (pathlib.Path(outdir) / f"{group}.json").write_text(json.dumps(results, indent=1))


# ---- the test ------------------------------------------------------------------------------------------------------

TRACE = re.compile(r"^\[jade\] (\S+) grid")


@pytest.mark.parametrize("group", GROUPS)
def test_paths_against_float64(group, tmp_path):
    env = dict(os.environ, JADE_TRACE_LAUNCH="1")
    for k in SWITCHES:
        env.pop(k, None)
    env.update(GROUP_ENV.get(group, {}))
    p = subprocess.run([sys.executable, str(pathlib.Path(__file__).resolve()), group, str(tmp_path)], env=env, cwd=str(ROOT),
                       capture_output=True, text=True, timeout=840)
    (tmp_path / "stderr.txt").write_text(p.stderr)
    assert p.returncode == 0, f"child exited {p.returncode}:\n{p.stderr[-4000:]}"
    seen, row = {}, None
    for line in p.stderr.splitlines():
        if line.startswith("[row] "):
            row = line[6:]
        m = TRACE.match(line)
        if m and row is not None:
            seen.setdefault(row, set()).add(m.group(1))
    results = json.loads((tmp_path / f"{group}.json").read_text())
    lines, errors = [], []
    for r in [r for r in ROWS if r["group"] == group]:
        missing = set(r["expect"]) - seen.get(r["name"], set())
        if missing:
            errors.append(f"{r['name']}: instantiations not launched: {sorted(missing)} (launched {sorted(seen.get(r['name'], []))})")
    for rec in results:
        if rec["error"]:
            errors.append(f"{rec['row']}: {rec['error']}")
        w = {k: max([l[k] for l in rec["launches"]] or [0.0]) for k in ("frac", "ddb")}
        lines.append(f"{rec['row']:<40} {len(rec['launches']):3d} checks  bound used {w['frac']:.3f}  |ddB| {w['ddb']:.1e}  "
                     f"pixels differing {sum(l['pixels_differing'] for l in rec['launches'])}  {rec['info']}")
    print("\n".join(lines))
    assert not errors, "\n".join(errors)


if __name__ == "__main__":
    _run_group(sys.argv[1], sys.argv[2])
