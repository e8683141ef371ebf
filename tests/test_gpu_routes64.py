"""Every kernel instantiation the engine can pick, against the float64 reference (tests/ref64.py), dB values and pixels.

One row per instantiation family: a configuration, launches that force each of its instantiations (dB-storing and
pixel-only, 16-byte aligned input, 8- but not 16-byte aligned input, unaligned input, long launches for the tensor-memory
ring forms, u8 palettes over several value ranges) and the inputs of ref64.standard_kinds: levels from 1 down to 3e-7 with
silent and subnormal stretches in the middle of the streams, a cosine at every bin (DC and Nyquist included), a unit
impulse at every frame offset, the stereo identities (one channel silent, L = R, L = -R, R = 1e-6 L) and loud inputs.
Rows with power_scale 1 / N^2 as well put the same inputs near the 1e-11 floor.

Which instantiation ran is read from the engine's launch trace (JADE_TRACE_LAUNCH: one `[jade] <kernel>[+run][+db][+u8]`
line per launch on stderr; the switch is read once per process), so each group of rows runs in a child process and the
test asserts that every instantiation its rows name was launched.

Not covered here: pkcta2<16> and pk2048x2, reachable only through the JADE_N65536 / JADE_PK_LOAD experiment switches.
"""
import json
import os
import pathlib
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = pathlib.Path(__file__).resolve().parent.parent

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

U8_RANGES = [(-50.0, 50.0), (-80.0, 0.0), (-120.0, 60.0), (0.0, 60.0), (58.0, 59.0)]
JADE = ("jade", 256, -50.0, 50.0)
NOT_U8 = ("jade", 255, -50.0, 50.0)  # not 256 colours: the pixel-only forms with the integer index clamp
# launches: (want_db, input offset in floats: 0 = 16-byte aligned, 2 = 8-byte aligned, 1 = unaligned, palette)
PACKED = [(True, 0, JADE), (False, 0, JADE), (True, 1, JADE)]
GENERAL = [(True, 0, JADE), (False, 0, JADE)]


def _row(name, group, cfg, expect, launches=PACKED, ps=(1.0, "1/N^2"), min_frames=0):
    return dict(name=name, group=group, cfg=cfg, expect=expect, launches=launches, ps=ps, min_frames=min_frames)


def _rows():
    R = []
    # pksmall<T>: one channel and a 2^n-channel sum, TMA-staged (dB-storing and pixel-only) and guarded
    for N, T in ((128, 2), (256, 4), (512, 8), (1024, 16)):
        for ch in (1, 2) if T != 8 else (1, 4):
            R.append(_row(f"pksmall<{T}> ch{ch}", "small", dict(fft_size=N, hop=N // 4, channels=ch),
                          [f"pksmall<{T}>+db", f"pksmall<{T}>", f"pksmall<{T}>-guard"]))
    # pk2048: one channel (and a four-channel sum), cp.async staging, LDG (8-byte aligned), guarded; the ring forms
    for ch in (1, 4):
        R.append(_row(f"pk2048 ch{ch}", "pk2048", dict(fft_size=2048, hop=512, channels=ch),
                      ["pk2048+db", "pk2048", "pk2048-guard", "pk2048-ldg+db", "pk2048-ldg"],
                      launches=PACKED + [(True, 2, JADE), (False, 2, JADE)]))
    for hop in (256, 512):
        R.append(_row(f"pk2048 ring hop{hop}", "pk2048", dict(fft_size=2048, hop=hop, channels=1),
                      ["pk2048+run+db", "pk2048+run"], launches=[(True, 0, JADE), (False, 0, JADE)], min_frames=44000))
    # pkz2048: staged, guarded (8-byte aligned and unaligned), u8, ring, ring-dB, ring-u8
    R.append(_row("pkz2048", "pkz2048", dict(fft_size=2048, hop=512, channels=2),
                  ["pkz2048+db", "pkz2048+u8", "pkz2048", "pkz2048-guard"],
                  launches=PACKED + [(True, 2, JADE), (False, 0, NOT_U8)] + [(False, 0, ("jade", 256) + r) for r in U8_RANGES]))
    R.append(_row("pkz2048 ring", "pkz2048", dict(fft_size=2048, hop=512, channels=2),
                  ["pkz2048+run+db", "pkz2048+run+u8", "pkz2048+run"],
                  launches=[(True, 0, JADE), (False, 0, NOT_U8)] + [(False, 0, ("jade", 256) + r) for r in U8_RANGES[:3]],
                  min_frames=34000))
    # pk3<16384>: staged, guarded, u8
    R.append(_row("pk3<16384>", "n16384", dict(fft_size=16384, hop=4096, channels=1, window="blackmanharris"),
                  ["pk3<16384>+db", "pk3<16384>+u8", "pk3<16384>", "pk3<16384>-guard"],
                  launches=PACKED + [(False, 0, NOT_U8)] + [(False, 0, ("jade", 256) + r) for r in U8_RANGES[1:]]))
    # pkcta<R1>: one channel and a two-channel sum
    for N, R1 in ((4096, 2), (8192, 4), (16384, 8), (32768, 16)):
        for ch in (1, 2) if N != 16384 else (2,):
            R.append(_row(f"pkcta<{R1}> ch{ch}", "pkcta", dict(fft_size=N, hop=N // 4, channels=ch),
                          [f"pkcta<{R1}>+db", f"pkcta<{R1}>"], launches=GENERAL))
    # N = 65536: one contributing channel (pkcl3), two channels (pkcl65536: AbsMean, Max; identity and log rows)
    R.append(_row("pkcl3<65536>", "n65536", dict(fft_size=65536, hop=16384, channels=1), ["pkcl3<65536>"], launches=GENERAL))
    for mix in ("absmean", "max"):
        R.append(_row(f"pkcl65536 {mix}", "n65536", dict(fft_size=65536, hop=16384, channels=2, mix_mode=mix),
                      ["pkcl65536"], launches=GENERAL))
        R.append(_row(f"pkcl65536 {mix} log rows", "n65536",
                      dict(fft_size=65536, hop=16384, channels=2, mix_mode=mix, sample_rate=192000.0, row_map="log_maxpool",
                           rows=300, fmin=20.0, fmax=96000.0), ["pkcl65536"], launches=GENERAL, ps=(1.0,)))
    # general kernels, one row per trigger: precise dB, un-flipped rows, linear crop, log rows, Max / Min, three channels
    trig = [("precise", dict(db_precise=1)), ("noflip", dict(flip_y=0)),
            ("crop", dict(row_map="linear_crop", fmin=1000.0, fmax=8000.0)),
            ("log", dict(row_map="log_maxpool", rows=64, fmin=50.0, fmax=20000.0)),
            ("max", dict(channels=2, mix_mode="max")), ("min", dict(channels=2, mix_mode="min")), ("3ch", dict(channels=3))]
    warp = [(64, 1), (128, 2), (256, 4), (512, 8), (1024, 16), (2048, 32), (2048, 32)]
    cta = [(4096, 2), (8192, 4), (16384, 8), (32768, 16), (4096, 2), (8192, 4), (16384, 8)]
    for k, (t, kw) in enumerate(trig):
        for fam, (N, r) in (("warp", warp[k]), ("cta", cta[k])):
            cfg = dict(fft_size=N, hop=N // 4, channels=1)
            cfg.update(kw)
            R.append(_row(f"{fam}<{r}> {t}", "general", cfg, [f"{fam}<{r}>"], launches=GENERAL, ps=(1.0,)))
    R.append(_row("warp<1> plain", "general", dict(fft_size=64, hop=16, channels=1), ["warp<1>"], launches=GENERAL))
    return R


ROWS = _rows()
GROUPS = sorted({r["group"] for r in ROWS})


# ---- child process -------------------------------------------------------------------------------------------------

def _run_group(group, outdir):
    import torch

    import oracle_lib as O
    import ref64
    from jadespectrogram_b200 import Engine

    results = []
    cache = {}
    for row in [r for r in ROWS if r["group"] == group]:
        cfg_kw = dict(sample_rate=48000.0, window="hann", mix_mode="absmean")
        cfg_kw.update(row["cfg"])
        N, hop, ch = cfg_kw["fft_size"], cfg_kw["hop"], cfg_kw["channels"]
        extra = 0
        kinds = ref64.standard_kinds(ch, N, hop)
        n = ref64.stream_length(N, hop, -(-len(ref64.impulse_offsets(N, hop)) // 8))
        cols = n // hop + 1
        if row["min_frames"]:
            extra = max(0, -(-row["min_frames"] // cols) - len(kinds))
            kinds = ref64.standard_kinds(ch, N, hop, extra)
        key = (N, hop, ch, cfg_kw["window"], n, len(kinds))
        if key not in cache:
            x = ref64.batch(kinds, ch, N, hop, n)
            cache.clear()
            cache[key] = (x, {})
        x, powers = cache[key]
        S = x.shape[0]
        d_buf = torch.zeros(S * ch * n + 8, dtype=torch.float32, device="cuda")
        for ps in row["ps"]:
            psv = float(np.float32(1.0 / (N * N))) if ps == "1/N^2" else float(ps)
            print(f"[row] {row['name']} ps={ps}", file=sys.stderr, flush=True)
            rec = dict(row=row["name"], ps=str(ps), launches=[], error=None)
            results.append(rec)
            try:
                eng = Engine(0, power_scale=psv, **cfg_kw)
                cfg = eng.get_config()
                ncols = eng.columns_for(n)
                assert ncols == cols, (ncols, cols)
                refs = []
                for s in range(S):
                    pk = (s, cfg.window)
                    if pk not in powers:
                        c1 = eng.get_config()
                        c1.power_scale = 1.0
                        powers[pk] = ref64.channel_power(c1, x[s], 0, ncols)
                    refs.append(ref64.Ref(cfg, None, 0, ncols, power=powers[pk]))
                for want_db, off, pal in row["launches"]:
                    scheme, npal, pmin, pmax = pal
                    eng.set_palette_scheme(scheme, npal)
                    eng.set_value_range(pmin, pmax)
                    d_in = d_buf[off:off + S * ch * n]
                    d_in.copy_(torch.from_numpy(x.reshape(-1)).to("cuda"))
                    d_pix = torch.empty((S, ncols, eng.R), dtype=torch.int32, device="cuda")
                    d_db = torch.empty((S, ncols, eng.B), dtype=torch.float32, device="cuda") if want_db else None
                    eng.render_device(d_in.data_ptr(), S, n, ch * n, n, 0, ncols, d_pix.data_ptr(),
                                      d_db.data_ptr() if want_db else None)
                    eng.sync()
                    pix = d_pix.cpu().numpy().view(np.uint32)
                    db = d_db.cpu().numpy() if want_db else None
                    opal = O.Palette(npal, O.PAL[scheme])
                    worst = dict(frac=0.0, a=0.0, b=0.0, ddb=0.0)
                    ndiff = 0
                    for s in range(S):
                        label = f"{row['name']} ps={ps} db={want_db} off={off} range=({pmin},{pmax}) stream {s} {kinds[s]}"
                        if want_db:
                            e = ref64.check_db64(db[s], refs[s], label)
                            worst = {k: max(worst[k], e[k]) for k in worst}
                        ndiff += ref64.check_pixels64(pix[s], refs[s], opal, pmin, pmax, npal, label)
                    rec["launches"].append(dict(db=want_db, off=off, pal=list(pal), pixels_differing=ndiff, **worst))
                eng.close()
            except Exception as ex:  # noqa: BLE001 -- reported to the parent, which fails the test
                rec["error"] = f"{type(ex).__name__}: {ex}"
        del d_buf
    (pathlib.Path(outdir) / f"{group}.json").write_text(json.dumps(results, indent=1))


# ---- the test ------------------------------------------------------------------------------------------------------

TRACE = re.compile(r"^\[jade\] (\S+) grid")


@pytest.mark.parametrize("group", GROUPS)
def test_routes_against_float64(group, tmp_path):
    env = dict(os.environ, JADE_TRACE_LAUNCH="1")
    for k in ("JADE_PK_LOAD", "JADE_RUN_MIN", "JADE_N16384", "JADE_N65536", "JADE_MAX_GRID", "JADE_BLOCKS_PER_SM"):
        env.pop(k, None)
    p = subprocess.run([sys.executable, str(pathlib.Path(__file__).resolve()), group, str(tmp_path)], env=env, cwd=str(ROOT),
                       capture_output=True, text=True, timeout=840)
    (tmp_path / "stderr.txt").write_text(p.stderr)
    assert p.returncode == 0, f"child exited {p.returncode}:\n{p.stderr[-4000:]}"
    seen, row = {}, None
    for line in p.stderr.splitlines():
        if line.startswith("[row] "):
            row = line[6:].rsplit(" ps=", 1)[0]
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
            errors.append(f"{rec['row']} ps={rec['ps']}: {rec['error']}")
        w = {k: max([l[k] for l in rec["launches"]] or [0.0]) for k in ("frac", "a", "b", "ddb")}
        lines.append(f"{rec['row']:<28} ps={rec['ps']:<6} bound used {w['frac']:.3f}  a {w['a']:.2f}  b {w['b']:.2e}  "
                     f"|ddB| {w['ddb']:.1e}  pixels off-edge-free, differing {sum(l['pixels_differing'] for l in rec['launches'])}")
    print("\n".join(lines))
    assert not errors, "\n".join(errors)


if __name__ == "__main__":
    sys.path.insert(0, str(ROOT))
    sys.path.insert(0, str(ROOT / "tests"))
    _run_group(sys.argv[1], sys.argv[2])
