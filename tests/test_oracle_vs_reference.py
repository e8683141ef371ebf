"""The restated oracle against the reference's REAL code.

oracle/_ref/libjade_ref.so compiles the reference's Spectrogram.cpp and CColorpalette.cpp where they lie, against the
inert JUCE/TGM stubs of oracle/shim/ (oracle/Makefile).  Everything the reference itself contains on the hot path --
buildmem geometry, the six windows, framing / staging, the channel-mix switch, dB, the ring, getMem, and the
timerCallback pixel loops -- therefore runs as written by its author and must agree BIT FOR BIT with the restatement in
oracle/jade_oracle.cpp.  The one thing that is not the reference's is the FFT (`spectrum`, absent TGM library): both
sides use the oracle's float32 stand-in, so FFT parity stays unpinned (DESIGN.md section 3).

Each test is a scenario that returns, in call order, every value the comparison looks at.  Where oracle/_ref is built, the
oracle's sequence is compared live with the reference's.  Every checkout also compares it with the sequence stored in
tests/golden/oracle_vs_reference.npz (a sha256 per value).  The stored values are the ORACLE's outputs, recorded while the
reference sources were not available; they have not been checked against the compiled reference in this form.  The same
comparisons, made live, last passed with oracle/_ref built at commit 9f207f4, and the oracle and its inputs are unchanged
since.  tools/gen_golden.py regenerates the file from the compiled reference only.
"""
import ctypes as C
import functools
import hashlib
import pathlib

import numpy as np
import pytest

import oracle_lib as O
import signals

# also_gpu: CPU-only, but selected by a `-m gpu` run too (tests/conftest.py), so that its record holds the whole pin
pytestmark = pytest.mark.also_gpu

FS = 48000.0
GOLD_PATH = pathlib.Path(__file__).parent / "golden" / "oracle_vs_reference.npz"


@functools.cache
def _gold():
    return dict(np.load(GOLD_PATH))


def digest(value):
    """sha256 of a value's dtype, shape and bytes (bit-exact identity of floats)."""
    a = np.ascontiguousarray(value)
    return np.frombuffer(hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).digest(), np.uint8)


def _first_difference(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return f"{a.dtype}{a.shape} vs {b.dtype}{b.shape}"
    bad = np.flatnonzero((a.reshape(-1).view(np.uint8).reshape(a.size, -1) != b.reshape(-1).view(np.uint8).reshape(b.size, -1)).any(1))
    return f"{bad.size} elements differ, the first at flat index {bad[0]}: {a.flat[bad[0]]!r} vs {b.flat[bad[0]]!r}"


def _pin(key, scenario):
    got = scenario(False)
    if O.have_ref_spec():
        live = scenario(True)
        assert [lab for lab, _ in live] == [lab for lab, _ in got]
        for (label, v), (_, r) in zip(got, live):
            assert np.array_equal(digest(v), digest(r)), f"{key}: {label} differs from the live reference: {_first_difference(v, r)}"
    want = _gold()[key]
    assert len(got) == len(want), (key, len(got), len(want))
    for i, ((label, v), d) in enumerate(zip(got, want)):
        assert np.array_equal(digest(v), d), f"{key}: value {i} ({label}) differs from the stored one"


def _spec(use_ref, N, feed, ch, fs=FS, mem_s=0.25, window="hann", mix=None):
    s = O.Spec(use_ref=use_ref)
    # the plugin's order (PluginProcessor.cpp:108-112)
    s.set_samplerate(fs)
    s.set_memory_time_s(mem_s)
    s.set_channels(ch)
    s.set_fftsize(N)
    s.set_feed_percent(O.FEED[feed])
    s.set_window(O.WIN[window])
    if mix is not None:
        s.set_mix_mode(O.MIX[mix])
    return s


def window_tables(window, N):
    def run(use_ref):
        if not use_ref:
            return [("window", O.window(window, N))]
        r = O.Spec(use_ref=True)
        r.set_fftsize(N)
        r.set_window(O.WIN[window])
        w = np.empty(N, np.float32)
        assert O.ref().jr_spec_window(r.h, w, N) == 0
        return [("window", w)]
    return run


def geometry_and_columns(feed, N, ch):
    def run(use_ref):
        s = _spec(use_ref, N, feed, ch)
        out = [(name, getattr(s, name)()) for name in ("spectrum_size", "memory_size", "feed_samples", "feed_blocks")]
        W, B = s.memory_size(), s.spectrum_size()
        x = signals.streams(1, ch, N * 9, FS, kind="mix", seed=N + ch)[0]
        mem = np.zeros((W, B), np.float32)
        # the first getMem reports "everything new" (int(100000000000), Spectrogram.cpp:18,168) and hands out the -120 ring
        out += [("first get_mem", s.get_mem(mem)), ("first ring", mem.copy())]
        assert (mem == -120.0).all()
        for b in range(9):
            out.append((f"process {b}", s.process(x[:, b * N:(b + 1) * N])))
            if b % 2 == 1 or b == 8:
                out += [(f"get_mem after block {b}", s.get_mem(mem)), (f"ring after block {b}", mem.copy())]
        return out
    return run


def mix_modes(mix):
    def run(use_ref):
        s = _spec(use_ref, 512, "p50", 2, mix=mix)
        W, B = s.memory_size(), s.spectrum_size()
        x = signals.streams(1, 2, 512 * 4, FS, kind="mix", seed=3)[0]
        x[1] *= 0.25
        mem = np.zeros((W, B), np.float32)
        for b in range(4):
            s.process(x[:, b * 512:(b + 1) * 512])
        return [("get_mem", s.get_mem(mem)), ("ring", mem)]
    return run


def pause_ring_wrap_and_setwindow_midstream(use_ref):
    s = _spec(use_ref, 256, "p25", 1, mem_s=0.02)  # a tiny ring: wraps several times
    W, B = s.memory_size(), s.spectrum_size()
    x = signals.streams(1, 1, 256 * 16, FS, kind="mix", seed=11)[0]
    mem = np.zeros((W, B), np.float32)
    s.get_mem(mem)
    out = []
    for b in range(16):
        if b == 5:
            s.set_pause(1)
        if b == 8:
            s.set_pause(0)
        if b == 10:
            s.set_window(O.WIN["flattop"])
        s.process(x[:, b * 256:(b + 1) * 256])
        if b in (2, 6, 9, 15):
            out += [(f"get_mem {b}", s.get_mem(mem)), (f"ring {b}", mem.copy())]
    out.append(("oversized get_mem", s.get_mem(np.zeros((W + 1, B), np.float32))[0]))
    assert out[-1][1] == -1
    return out


def next_pow2_and_ms_setter(use_ref):
    s = O.Spec(use_ref=use_ref)
    out = []
    for fs in (44100.0, 48000.0, 96000.0):
        s.set_samplerate(fs)
        for ms in (1.0, 5.0, 10.7, 21.3, 42.7, 100.0):
            out.append((f"next_pow2 {fs} {ms}", s.next_pow2(ms)))
            s.set_closest_fftsize_ms(ms)
            out.append((f"sizes {fs} {ms}", (s.spectrum_size(), s.memory_size())))
    return out


def timer_callback_pixel_loops(running):
    """SpectrogramComponent::timerCallback as written (Spectrogram.cpp:590-731) vs the restated view, pixel for pixel."""
    def run(use_ref):
        N = 256
        s = _spec(use_ref, N, "p50", 2, mem_s=0.1)
        v = O.View(s, use_ref=True) if use_ref else O.View(s, O.Palette(256, O.PAL["jade"]))
        v.set_running(running)
        x = signals.streams(1, 2, N * 14, FS, kind="mix", seed=5)[0]
        v.tick()  # full redraw of the -120 ring
        out = [("first image", v.image())]
        W = s.memory_size()
        done = 0
        for nblk in (1, 3, 2, 1):
            for _ in range(nblk):
                s.process(x[:, done * N:(done + 1) * N])
                done += 1
            v.tick()
            if not running:
                # The reference draws its red cursor at pos+dd and only wraps the == W case (Spectrogram.cpp:713-716), i.e. it
                # writes out of bounds when pos+dd > W; the restatement wraps.  Compare away from that corner.
                pos = (done * 2) % W
                if pos + 4 > W:
                    continue
            out.append((f"image after {done} blocks", v.image()))
        # range change -> m_recomputeAll (Spectrogram.cpp:370,379,623-657)
        v.set_color_range(-80.0, 10.0)
        v.tick()
        out.append(("image after range change", v.image()))
        return out
    return run


def bench_entry_point_frames(use_ref):
    """Frames counted by the CPU baseline's batch entry point (reference glue, or the oracle port bench.py falls back to)."""
    x = signals.streams(1, 2, 2048 * 6, FS, kind="mix")[0]
    frames = C.c_long(0)
    if use_ref:
        fps = O.ref().jr_bench_batch(FS, 2048, O.FEED["p25"], O.WIN["hann"], 2, O.PAL["jade"], 256, -50.0, 50.0, x.reshape(-1),
                                     x.shape[1], 4, 2, C.byref(frames))
    else:
        cfg = O.BatchCfg(FS, 2048, 512, O.WIN["hann"], 2, O.MIX["absmean"], O.PAL["jade"], 256, 0, -50.0, 50.0, 0)
        fps = O.lib().jo_bench_batch(C.byref(cfg), x.reshape(-1), x.shape[1], 4, 2, C.byref(frames))
    assert fps > 0
    return [("frames", frames.value)]


WINDOW_NS = [64, 512, 2048, 16384, 65536]
GEOMETRIES = [(256, 1), (1024, 2), (2048, 2)]


def scenarios():
    """golden key -> scenario, for tools/gen_golden.py."""
    out = {f"window_{w}_{n}": window_tables(w, n) for w in O.WIN for n in WINDOW_NS}
    out.update({f"geometry_{f}_{n}_{c}": geometry_and_columns(f, n, c) for f in O.FEED for n, c in GEOMETRIES})
    out.update({f"mix_{m}": mix_modes(m) for m in O.MIX})
    out.update(pause=pause_ring_wrap_and_setwindow_midstream, next_pow2=next_pow2_and_ms_setter,
               timer_1=timer_callback_pixel_loops(1), timer_0=timer_callback_pixel_loops(0), bench_frames=bench_entry_point_frames)
    return out


@pytest.mark.parametrize("window", list(O.WIN))
@pytest.mark.parametrize("N", WINDOW_NS)
def test_window_tables(window, N):
    _pin(f"window_{window}_{N}", window_tables(window, N))


@pytest.mark.parametrize("feed", list(O.FEED))
@pytest.mark.parametrize("N,ch", GEOMETRIES)
def test_geometry_and_columns(feed, N, ch):
    _pin(f"geometry_{feed}_{N}_{ch}", geometry_and_columns(feed, N, ch))


@pytest.mark.parametrize("mix", list(O.MIX))
def test_mix_modes(mix):
    _pin(f"mix_{mix}", mix_modes(mix))


def test_pause_ring_wrap_and_setwindow_midstream():
    _pin("pause", pause_ring_wrap_and_setwindow_midstream)


def test_next_pow2_and_ms_setter():
    _pin("next_pow2", next_pow2_and_ms_setter)


@pytest.mark.parametrize("running", [1, 0])
def test_timer_callback_pixel_loops(running):
    _pin(f"timer_{running}", timer_callback_pixel_loops(running))


def test_reference_bench_entry_point_counts_frames():
    _pin("bench_frames", bench_entry_point_frames)
    assert bench_entry_point_frames(False) == [("frames", 4 * 6 * 4)]
