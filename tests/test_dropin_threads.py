"""Thread-safety and source-compatibility of the drop-in C++ boundary, checked WITHOUT a GPU:
  * include/Spectrogram.h under ThreadSanitizer: audio thread (re-blocker -> processSynchronBlock) against the GUI thread
    (getMem, setWindow, setPauseMode, structural setters), linked with a CPU fake of the C ABI (tests/dropin/fake_jade_gpu.cpp
    -- test infrastructure, computes nothing);
  * the JUCE / TGM branch of the header (SpectrogramParameter, prepareParameter, Spectrogram.h:22-76,113; call site
    PluginProcessor.cpp:28) compiles against the inert stubs in oracle/shim."""
import pathlib
import subprocess

import pytest

ROOT = pathlib.Path(__file__).resolve().parent.parent


def _run(cmd, **kw):
    return subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, **kw)


def test_dropin_class_is_race_free_under_tsan(tmp_path):
    exe = tmp_path / "tsan_dropin"
    r = _run(["g++", "-std=c++17", "-O1", "-g", "-fsanitize=thread", "-pthread", "-I", "include", "tests/dropin/tsan_dropin.cpp",
              "tests/dropin/fake_jade_gpu.cpp", "-o", str(exe)])
    if r.returncode != 0 and "sanitize" in r.stderr:
        pytest.skip("ThreadSanitizer runtime not available: " + r.stderr[-200:])
    assert r.returncode == 0, r.stderr[-2000:]
    r = _run([str(exe)], timeout=600)
    assert "ThreadSanitizer" not in r.stderr, r.stderr[-3000:]
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout[-1000:] + r.stderr[-1000:]
    assert " 0 errors" in r.stdout


def test_plugin_shell_compiles_against_the_dropin_header():
    r = _run(["g++", "-std=c++17", "-fsyntax-only", "-Wall", "-I", "include", "-I", "oracle/shim", "tests/dropin/plugin_compile_test.cpp"])
    assert r.returncode == 0, r.stderr[-3000:]
