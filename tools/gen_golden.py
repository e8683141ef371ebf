#!/usr/bin/env python3
"""Generate the committed golden fixtures under tests/golden/ (run in the build container, where /root/reference exists).

  palette_ref.npz  -- colour tables and lookup sweeps produced by the REFERENCE's own CColorpalette.cpp compiled in place
                      (oracle/_ref/libjade_ref.so): 7 schemes x {2,3,7,64,255,256,1024} colours x invert {0,1}, plus
                      getRGBColor sweeps over several value ranges (incl. >=max, <min, max<=0, equal bounds).
  windows.npz      -- the six unit-RMS window tables at N = 64 and 2048 from the oracle restatement of setWindowFkt
                      (Spectrogram.cpp:239-293), and sha256 digests at N = 65536.
  pipeline.npz     -- seeded inputs with the oracle's dB columns and ARGB pixels for small end-to-end cases.
  spectrogram_ref.npz -- outputs of the REFERENCE's own Spectrogram class and SpectrogramComponent::timerCallback
                      (Spectrogram.cpp compiled in place against the stub JUCE/TGM headers of oracle/shim/, FFT = the
                      oracle's float32 stand-in): window tables, dB rings after streaming seeded blocks through
                      processSynchronBlock/getMem for every feed percentage, and the assembled image.

  paint_ref.npz    -- what the REFERENCE's own SpectrogramComponent::paint draws (crop rectangle of the spectrogram blit, the
                      tick values / label boxes of both axes, the colourbar pixels) for a few sizes and slider positions.
  oracle_vs_reference.npz -- the reference's side of every comparison in tests/test_oracle_vs_reference.py (sha256 per value;
                      the committed file holds the oracle's side, see that test's docstring).

    python tools/gen_golden.py          (everything)      python tools/gen_golden.py paint   (paint_ref.npz only)
    python tools/gen_golden.py oracle_vs_reference        (oracle_vs_reference.npz only)
"""
import hashlib
import pathlib
import sys

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
import oracle_lib as O  # noqa: E402
import signals  # noqa: E402

OUT = ROOT / "tests" / "golden"
OUT.mkdir(exist_ok=True)

SIZES = (2, 3, 7, 64, 255, 256, 1024)
RANGES = [(-50.0, 50.0), (0.0, 1.0), (-120.0, -20.0), (-80.0, 0.0), (10.0, -10.0), (-30.0, -30.0), (5.0, 5.0), (0.0, 0.0)]


def sweep_values(mn, mx):
    lo, hi = min(mn, mx), max(mn, mx)
    span = max(hi - lo, 1.0)
    v = np.linspace(lo - 0.25 * span, hi + 0.25 * span, 4001).astype(np.float32)
    extra = np.array([lo, hi, np.nextafter(np.float32(hi), np.float32(-1e9)), np.float32(hi) * np.float32(0.9999), -1e30, 1e30],
                     np.float32)
    return np.concatenate([v, extra])


def palettes():
    assert O.ref() is not None, "oracle/_ref/libjade_ref.so missing: run `make -C oracle` where /root/reference exists"
    out = {}
    for scheme in range(7):
        for n in SIZES:
            for inv in (0, 1):
                p = O.Palette(n, scheme, use_ref=True)
                if inv:
                    p.set_invert(1)
                    p.set_color_scheme(scheme)
                out[f"table_s{scheme}_n{n}_i{inv}"] = p.table().astype(np.int32)
    # stale-entry quirk: kMono+invert after another scheme keeps the upper half of the previous table
    p = O.Palette(256, 6, use_ref=True)
    p.set_invert(1)
    p.set_color_scheme(0)
    out["table_jade_then_mono_inverted_n256"] = p.table().astype(np.int32)
    p = O.Palette(None, None, use_ref=True)
    out["table_default_ctor"] = p.table().astype(np.int32)
    for i, (mn, mx) in enumerate(RANGES):
        for n, scheme in ((256, 6), (64, 4), (7, 3)):
            p = O.Palette(n, scheme, use_ref=True)
            p.set_value_range(mn, mx)
            v = sweep_values(mn, mx)
            # the reference's own range rules (CColorpalette.cpp:39-54); m_Min >= m_Max (equal non-positive bounds) makes
            # its index negative / NaN, i.e. an out-of-bounds read: those ranges have no defined reference output
            a, b = np.float32(min(mn, mx)), np.float32(max(mn, mx))
            if a == b:
                a = np.float32(0.99 * float(b))
            if not (b > a):
                continue
            out[f"sweep_values_r{i}_n{n}_s{scheme}"] = v
            out[f"sweep_colors_r{i}_n{n}_s{scheme}"] = p.lookup(v).astype(np.int32)
    np.savez_compressed(OUT / "palette_ref.npz", **out)
    print("palette_ref.npz", len(out), "arrays")


def windows():
    out = {}
    for name in O.WIN:
        for n in (64, 2048):
            out[f"{name}_{n}"] = O.window(name, n)
        out[f"{name}_65536_sha256"] = np.frombuffer(hashlib.sha256(O.window(name, 65536).tobytes()).digest(), np.uint8)
    np.savez_compressed(OUT / "windows.npz", **out)
    print("windows.npz", len(out), "arrays")


def pipeline():
    out = {}
    cases = [("n64_mono", 64, 16, 1, "hann", "absmean"), ("n256_stereo", 256, 64, 2, "blackmanharris", "absmean"),
             ("n1024_cfg1", 1024, 512, 1, "hann", "absmean"), ("n2048_cfg2", 2048, 512, 2, "hann", "absmean"),
             ("n512_max3", 512, 128, 3, "hamming", "max")]
    for name, N, hop, ch, win, mix in cases:
        ncols = 12
        x = signals.streams(1, ch, hop * ncols, 48000.0, kind="mix", seed=7 + N)[0]
        db, pix = O.render_batch(x, fft_size=N, hop=hop, window=win, mix=mix, ncols=ncols + 1)
        out[name + "_x"] = x
        out[name + "_db"] = db
        out[name + "_pix"] = pix
        out[name + "_cfg"] = np.array([N, hop, ch, O.WIN[win], O.MIX[mix]], np.int32)
    np.savez_compressed(OUT / "pipeline.npz", **out)
    print("pipeline.npz", len(out), "arrays")


REF_CASES = [("n256_p100_mono", 256, "p100", 1, "hann", 6), ("n512_p50_stereo", 512, "p50", 2, "blackmanharris", 5),
             ("n1024_p25_stereo", 1024, "p25", 2, "hann", 4), ("n512_p10_mono", 512, "p10", 1, "hannpoisson", 4)]


def ref_case_inputs(N, ch, nblocks):
    return signals.streams(1, ch, N * nblocks, 48000.0, kind="mix", seed=100 + N + ch)[0]


def reference_class():
    assert O.have_ref_spec(), "oracle/_ref/libjade_ref.so lacks the Spectrogram glue: run `make -C oracle`"
    out = {}
    for name in O.WIN:  # the real setWindowFkt (Spectrogram.cpp:239-293)
        for n in (64, 1024):
            r = O.Spec(use_ref=True)
            r.set_fftsize(n)
            r.set_window(O.WIN[name])
            w = np.empty(n, np.float32)
            assert O.ref().jr_spec_window(r.h, w, n) == 0
            out[f"window_{name}_{n}"] = w
    for name, N, feed, ch, win, nblocks in REF_CASES:
        r = O.Spec(use_ref=True)
        r.set_samplerate(48000.0)
        r.set_memory_time_s(0.1)
        r.set_channels(ch)
        r.set_fftsize(N)
        r.set_feed_percent(O.FEED[feed])
        r.set_window(O.WIN[win])
        W, B = r.memory_size(), r.spectrum_size()
        view = O.View(r, use_ref=True)
        view.tick()
        x = ref_case_inputs(N, ch, nblocks)
        mem = np.zeros((W, B), np.float32)
        for b in range(nblocks):
            r.process(x[:, b * N:(b + 1) * N])
        view.tick()
        img = view.image()
        for b in range(nblocks):  # second pass so that getMem below sees exactly these columns again
            r.process(x[:, b * N:(b + 1) * N])
        newvals, pos = r.get_mem(mem)
        out[name + "_cfg"] = np.array([N, O.FEED[feed], ch, O.WIN[win], nblocks, W, B, newvals, pos], np.int32)
        out[name + "_ring_db"] = mem
        out[name + "_image"] = img
    np.savez_compressed(OUT / "spectrogram_ref.npz", **out)
    print("spectrogram_ref.npz", len(out), "arrays")


# (component width, height, m_scaleFactor, min Hz, max Hz, fs, FFT size, colour scheme, colour range)
PAINT_CASES = [
    (800, 550, 1.0, 1.0, 20000.0, 48000.0, 2048, 6, (-50.0, 50.0)),
    (800, 550, 1.0, 100.0, 8000.0, 48000.0, 2048, 6, (-50.0, 50.0)),
    (1100, 756, 1.375, 37.5, 12345.0, 44100.0, 1024, 4, (-30.0, 20.0)),
    (1400, 962, 1.75, 500.0, 30000.0, 48000.0, 4096, 2, (-50.0, 0.0)),     # max above fs/2: clamped
    (800, 550, 1.0, 9000.0, 600.0, 96000.0, 8192, 5, (10.0, -10.0)),        # min above max: 0.9 max
    (937, 611, 1.17, 20.0, 149.0, 48000.0, 512, 1, (-80.0, -20.0)),        # ticks below the 150 Hz rounding rule
]


def paint_reference():
    """The reference's own SpectrogramComponent::paint (oracle/_ref, recording Graphics stub): crop rectangle, axis ticks and
    colourbar for a few component sizes / slider positions -> tests/golden/paint_ref.npz."""
    assert O.have_ref_spec() and hasattr(O.ref(), "jr_view_paint"), "rebuild oracle/_ref (`make -C oracle`)"
    out = {"cases": np.array([[c[0], c[1], c[2], c[3], c[4], c[5], c[6], c[7], c[8][0], c[8][1]] for c in PAINT_CASES], np.float64)}
    for i, (w, h, scale, lo, hi, fs, N, scheme, rng) in enumerate(PAINT_CASES):
        r = O.Spec(use_ref=True)
        r.set_samplerate(fs)
        r.set_memory_time_s(0.1)
        r.set_fftsize(N)
        view = O.View(r, use_ref=True)
        view.set_scheme(scheme)
        view.set_color_range(*rng)
        view.tick()  # sizes the internal image (m_internalHeight = bins) and applies the colour range
        p = view.paint(w, h, scale, lo, hi)
        out[f"c{i}_crop"] = np.array(p["crop"], np.int32)
        out[f"c{i}_hz"] = np.array([p["min_hz"], p["max_hz"]], np.float32)
        for k in ("freq_val", "freq_y", "color_val", "color_y", "colorbar"):
            out[f"c{i}_{k}"] = p[k]
    np.savez_compressed(OUT / "paint_ref.npz", **out)
    print("paint_ref.npz", len(out), "arrays")


def oracle_vs_reference():
    """tests/golden/oracle_vs_reference.npz: what the compiled reference returns in each scenario of
    tests/test_oracle_vs_reference.py (a sha256 per value)."""
    assert O.have_ref_spec(), "oracle/_ref/libjade_ref.so lacks the Spectrogram glue: run `make -C oracle` where the reference exists"
    import test_oracle_vs_reference as T
    out = {key: np.stack([T.digest(v) for _, v in run(True)]) for key, run in T.scenarios().items()}
    np.savez_compressed(OUT / "oracle_vs_reference.npz", **out)
    print("oracle_vs_reference.npz", len(out), "arrays")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "oracle_vs_reference":
        oracle_vs_reference()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "paint":
        paint_reference()
        sys.exit(0)
    palettes()
    windows()
    pipeline()
    reference_class()
    paint_reference()
    oracle_vs_reference()
