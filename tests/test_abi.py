"""C-ABI + host-logic checks that need no GPU: the shared library loads, exports
every symbol include/*.h declares, the host-only helpers agree with the oracle,
and every compute entry point fails loudly (no CPU fallback) without a device."""
import ctypes as C
import glob
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    names = set()
    for h in glob.glob(os.path.join(ROOT, "include", "*.h")):
        src = re.sub(r"/\*.*?\*/", "", open(h).read(), flags=re.S)
        names |= set(re.findall(r"\b(vp_[a-z0-9_]+)\s*\(", src))
    return names


def test_library_exports_every_declared_symbol(vp):
    lib = vp.load_library()
    decl = declared_symbols()
    assert len(decl) >= 26
    for name in sorted(decl):
        assert hasattr(lib, name), "libvp_engine.so does not export %s" % name
    assert decl == set(vp.ABI_SYMBOLS)


def test_struct_layouts_match_header(vp):
    assert C.sizeof(vp.Params) == 40 and C.sizeof(vp.Sizes) == 13 * 4
    assert C.sizeof(vp.PitchFrame) == 4 * 10 + 4 * 2 * vp.VP_MAX_MARKS + 8 == 240


def test_default_params_are_the_plugin_defaults(vp):
    p = vp.default_params()  # PluginProcessor.cpp:37-73
    assert (p.gainPitch, p.gainVoice, p.gainSynth, p.gainVoc) == (0.0, -60.0, -60.0, 0.0)
    assert (p.lpcVoice, p.lpcPitch, p.lpcSynth, p.keyPitch, p.pitchBool, p.vocBool) == (40, 15, 5, 12, 1, 1)


@pytest.mark.parametrize("fs,B,key", [(44100.0, 1024, 12), (48000.0, 1024, 3), (44100.0, 128, 0), (96000.0, 512, 12),
                                      (22050.0, 64, 5)])
def test_sizes_agree_with_oracle(vp, oracle, fs, B, key):
    a, b = vp.sizes_for(fs, B, key), oracle.sizes_for(fs, B, key)
    for k in b:
        assert a[k] == b[k], k
    assert a["tauMin"] == int(np.floor(fs / 800.0))


def test_bad_arguments_are_codes_not_crashes(vp):
    lib = vp.load_library()
    s = vp.Sizes()
    assert lib.vp_sizes_for(44100.0, 0, 12, C.byref(s)) == vp.VP_E_ARG
    assert lib.vp_sizes_for(44100.0, 1024, 13, C.byref(s)) == vp.VP_E_ARG
    assert lib.vp_sizes_for(44100.0, 1024, 12, None) == vp.VP_E_ARG
    assert lib.vp_engine_prepare(None, 44100.0, 1024, 1, 1, 0) == vp.VP_E_ARG
    assert lib.vp_engine_sync(None) == vp.VP_E_ARG
    assert lib.vp_engine_process_device(None, 1, None, None, None, None, None, 0) == vp.VP_E_ARG
    assert lib.vp_synth_host(44100.0, 0, 0, 0, 16, 16, None, None, None) == vp.VP_E_ARG
    assert lib.vp_last_error(None) == b"null engine"
    assert lib.vp_stage_name(0) == b"gate" and lib.vp_stage_name(99) == b""


NO_DEVICE_CHECK = """
import ctypes as C
import sys
sys.path.insert(0, %r)
import vocoderproject_b200 as vp
lib = vp.load_library()
assert lib.vp_device_count() == 0, lib.vp_device_count()
h = C.c_void_p()
assert lib.vp_engine_create(C.byref(h), 0) == vp.VP_E_CUDA and not h.value
try:
    vp.Engine(44100.0, 1024, 1, 4)
except vp.EngineError as ex:
    assert ex.code == vp.VP_E_CUDA, ex.code
else:
    raise AssertionError("an engine was created without a device")
"""


def test_no_cpu_fallback_without_a_device(vp):
    """In a child process that sees no CUDA device (CUDA_VISIBLE_DEVICES empty), so that it holds on a GPU machine too."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, "-c", NO_DEVICE_CHECK % ROOT], env=env, capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stdout + res.stderr


def test_missing_library_fails_loudly(vp, tmp_path):
    with pytest.raises(vp.EngineError):
        vp.load_library(str(tmp_path / "nope.so"))


def test_product_package_never_touches_the_oracle():
    """oracle/ is test infrastructure: nothing under the package may import, link or call it."""
    pkg = os.path.join(ROOT, "vocoderproject_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp")):
                src = open(os.path.join(dirpath, f), errors="replace").read()
                assert "oraclebind" not in src and "refbind" not in src and "vp_oracle" not in src and \
                    "libvpref" not in src, os.path.join(dirpath, f)


def test_synth_host_is_deterministic_and_stream_indexed(vp):
    a = vp.synth_host(44100.0, 3, 4096, flavour=0, first_stream=10)
    b = vp.synth_host(44100.0, 1, 4096, flavour=0, first_stream=11)
    assert np.array_equal(a[0][1], b[0][0]) and np.array_equal(a[1][1], b[1][0]) and np.array_equal(a[2][1], b[2][0])
    assert not np.array_equal(a[0][0], a[0][1])
    assert 0.2 < np.abs(a[0]).max() < 1.0 and np.abs(a[1]).max() <= 0.26
    clean = vp.synth_host(44100.0, 1, 4096, flavour=1, first_stream=10)
    assert np.abs(clean[0][0] - a[0][0]).max() < 0.05  # same voice, lower aspiration noise
