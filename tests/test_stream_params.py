"""Per-stream key and gains (vp_stream_params, vp_engine_set_stream_params): each stream of a batch is its own plug-in
instance with its own parameter tree.

CPU: the struct layout matches the header, the entry points refuse null arguments.
GPU: a batch with per-stream values equals, bit for bit, every stream run alone with vp_engine_set_params; it matches the
reference run with each stream's own values (also under per-stream automation, in streaming, in defined mode and on the
host paths); the broadcast, getter, reset, asynchronous and error semantics of the header hold."""
import ctypes as C
import json
import os
import shutil
import subprocess

import numpy as np
import pytest

import refbind
from common import MAXABS_MAX, SNR_MIN_DB, assert_decisions, compare_decisions, maxabs, oracle_decisions, reference_runs, snr_db

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("gainPitch", "gainVoice", "gainSynth", "gainVoc", "keyPitch")

LAYOUT_PROBE = r"""
#include <stddef.h>
#include <stdio.h>
#include "vp_engine.h"
int main(void) {
    printf("%zu %zu %zu %zu %zu %zu\n", sizeof(vp_stream_params), offsetof(vp_stream_params, gainPitch),
           offsetof(vp_stream_params, gainVoice), offsetof(vp_stream_params, gainSynth), offsetof(vp_stream_params, gainVoc),
           offsetof(vp_stream_params, keyPitch));
    return 0;
}
"""


# ---------------------------------------------------------------------------------------------------------- CPU
def test_stream_params_layout_matches_header(vp, tmp_path):
    assert C.sizeof(vp.StreamParams) == 20
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler to read the header's layout")
    src = tmp_path / "probe.c"
    src.write_text(LAYOUT_PROBE)
    exe = str(tmp_path / "probe")
    subprocess.check_call([cc, "-I", os.path.join(ROOT, "include"), "-o", exe, str(src)])
    got = [int(x) for x in subprocess.check_output([exe], text=True).split()]
    assert got == [C.sizeof(vp.StreamParams)] + [getattr(vp.StreamParams, f).offset for f in FIELDS]


def test_stream_params_null_arguments_are_codes(vp):
    lib = vp.load_library()
    arr = (vp.StreamParams * 1)()
    assert lib.vp_engine_set_stream_params(None, 0, 1, arr) == vp.VP_E_ARG
    assert lib.vp_engine_get_stream_params(None, 0, 1, arr) == vp.VP_E_ARG
    assert vp.stream_params().as_dict() == dict(gainPitch=0.0, gainVoice=-60.0, gainSynth=-60.0, gainVoc=0.0, keyPitch=12)


# ---------------------------------------------------------------------------------------------------------- GPU helpers
def spread(S):
    """Per-stream values: keys 0..12 (twice for 26 streams), gains over the plug-in's range, the dry paths' switching
    point on both sides (-59.0 dB is off, -58.9 dB on), some streams with dry voice and / or dry side-chain."""
    voc = np.linspace(-24.0, 6.0, S)
    pitch = np.linspace(6.0, -30.0, S)
    items = []
    for s in range(S):
        it = dict(keyPitch=s % 13, gainVoc=float(voc[s]), gainPitch=float(pitch[s]), gainVoice=-60.0, gainSynth=-60.0)
        if s % 5 == 1:
            it["gainVoice"] = -59.0
        if s % 5 == 2:
            it["gainVoice"] = -58.9
        if s % 7 == 3:
            it["gainSynth"] = -12.0
        if s % 7 == 4:
            it["gainSynth"] = -59.0
        if s % 11 == 5:
            it["gainVoice"], it["gainSynth"] = -6.0, -58.9
        if s == S - 1:
            it["gainVoc"], it["gainPitch"] = -60.0, -59.5
        items.append(it)
    return items


def run_batch(vp, fs, B, voice, sl, sr, items, workspace_bytes=0):
    S, n = voice.shape
    eng = vp.Engine(fs, B, S, n // B, workspace_bytes=workspace_bytes)
    try:
        eng.set_stream_params(0, items)
        outL, outR = eng.process(voice, sl, sr)
        pf = [[bytes(f) for f in eng.pitch_frames(s)] for s in range(S)]
        vf = [eng.voc_frames(s) for s in range(S)]
        frames = [eng.pitch_frames(s) for s in range(S)]
        return dict(outL=outL, outR=outR, pf=pf, vf=vf, frames=frames, passes=-(-S // eng.info()["streams_per_pass"]))
    finally:
        eng.close()


def run_alone(vp, fs, B, voice, sl, sr, it):
    n = len(voice)
    eng = vp.Engine(fs, B, 1, n // B, params=vp.default_params(**it))
    try:
        outL, outR = eng.process(voice[None], sl[None], None if sr is None else sr[None])
        return dict(outL=outL[0], outR=outR[0], pf=[bytes(f) for f in eng.pitch_frames(0)], vf=eng.voc_frames(0))
    finally:
        eng.close()


def assert_same_stream(a, b, s, what):
    assert np.array_equal(a["outL"][s], b["outL"]), "%s: stream %d outL" % (what, s)
    assert np.array_equal(a["outR"][s], b["outR"]), "%s: stream %d outR" % (what, s)
    assert a["pf"][s] == b["pf"], "%s: stream %d pitch frame records" % (what, s)
    for k in ("gated", "EeVoice", "EeSynth", "g"):
        assert np.array_equal(a["vf"][s][k], b["vf"][k]), "%s: stream %d vocoder frames %s" % (what, s, k)


def assert_audio(ref, got, what):
    sn, mx = snr_db(ref, got), maxabs(ref, got)
    assert sn >= SNR_MIN_DB and mx <= MAXABS_MAX, "%s: SNR %.1f dB, max abs err %.3e" % (what, sn, mx)


def ref_run(fs, B, voice, sl, sr, params, schedule=None):
    """The reference's own C++ when it is built here, else the C oracle port (bit-identical to it)."""
    import oraclebind
    if refbind.available("strict"):
        return refbind.run(fs, B, voice, sl, synthR=sr, params=params, log=True, schedule=schedule)
    return oraclebind.run(fs, B, voice, sl, synthR=sr, params=params, log=True, schedule=schedule)


SECS = 6.0
B = 1024
S26 = 26


@pytest.fixture(scope="module", params=[44100.0, 48000.0], ids=["44k1", "48k"])
def batch(request, vp):
    fs = request.param
    n = int(fs * SECS) // B * B
    voice, sl, sr = vp.synth_host(fs, S26, n, flavour=0, first_stream=3000)
    items = spread(S26)
    return dict(fs=fs, voice=voice, sl=sl, sr=sr, items=items, res=run_batch(vp, fs, B, voice, sl, sr, items))


# ---------------------------------------------------------------------------------------------------------- GPU tests
@pytest.mark.gpu
def test_batch_equals_separate_instances_bitwise(vp, batch):
    """One engine with per-stream values == each stream alone in its own engine with vp_engine_set_params, bit for bit
    (outL, outR, every pitch and vocoder frame record); again with a workspace that forces several passes."""
    fs, voice, sl, sr, items, res = batch["fs"], batch["voice"], batch["sl"], batch["sr"], batch["items"], batch["res"]
    alone = [run_alone(vp, fs, B, voice[s], sl[s], sr[s], items[s]) for s in range(S26)]
    for s in range(S26):
        assert_same_stream(res, alone[s], s, "one pass")
    # streams with the dry side-chain on have their own right channel, the others L == R
    for s, it in enumerate(items):
        assert np.array_equal(res["outL"][s], res["outR"][s]) == (it["gainSynth"] <= -59.0), s
    # several passes: the table is read at streamBase + stream of the pass
    eng = vp.Engine(fs, B, S26, voice.shape[1] // B)
    per = eng.info()["workspace_bytes"] // S26
    eng.close()
    multi = run_batch(vp, fs, B, voice, sl, sr, items, workspace_bytes=7 * per + per // 2)
    assert multi["passes"] >= 3
    for s in range(S26):
        assert_same_stream(multi, alone[s], s, "%d passes" % multi["passes"])


@pytest.mark.gpu
def test_batch_matches_reference_per_stream(vp, batch):
    fs, voice, sl, sr, items, res = batch["fs"], batch["voice"], batch["sl"], batch["sr"], batch["items"], batch["res"]
    refs, kind = reference_runs([(fs, B, voice[s], sl[s], sr[s], items[s]) for s in range(S26)])
    for s in range(S26):
        what = "stream %d %r (%s)" % (s, items[s], kind)
        assert_audio(refs[s]["outL"], res["outL"][s], what + " L")
        assert_audio(refs[s]["outR"], res["outR"][s], what + " R")
        assert_decisions(compare_decisions(vp, oracle_decisions(refs[s]["pitch"]), res["frames"][s]), what)


@pytest.mark.gpu
def test_per_stream_automation(vp):
    """Different streams change key / gains at different process calls: each equals the reference run with its own
    schedule, and bit for bit a single-stream engine driven with vp_engine_set_params at the same cuts."""
    fs, S = 44100.0, 4
    nb = int(fs * SECS) // B
    voice, sl, sr = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=3100)
    base = [dict(keyPitch=12), dict(keyPitch=3, gainVoc=-6.0), dict(keyPitch=7, gainPitch=-3.0), dict(keyPitch=0)]
    changes = {  # block -> {stream: new values}
        60: {0: dict(keyPitch=5), 2: dict(keyPitch=10, gainPitch=2.0)},
        130: {1: dict(gainVoc=3.0, keyPitch=11), 3: dict(gainVoice=-20.0)},
        200: {2: dict(gainVoc=-12.0), 3: dict(keyPitch=8, gainSynth=-18.0), 0: dict(gainPitch=-9.0)},
    }
    cuts = [0, 60, 130, 200, nb]
    # per stream: the values in force from each cut on
    state = [dict(b) for b in base]
    per_cut = []
    for a in cuts[:-1]:
        for s, d in changes.get(a, {}).items():
            state[s].update(d)
        per_cut.append([dict(x) for x in state])
    eng = vp.Engine(fs, B, S, max(b - a for a, b in zip(cuts, cuts[1:])))
    outL, outR, pf = [], [], [[] for _ in range(S)]
    try:
        for c, (a, b) in enumerate(zip(cuts, cuts[1:])):
            if c == 0:
                eng.set_stream_params(0, per_cut[0])
            else:
                for s, d in changes[a].items():
                    eng.set_stream_params(s, [d])  # a partial dict keeps the stream's other values
            assert eng.stream_params() == [vp.stream_params(**x).as_dict() for x in per_cut[c]]
            l, r = eng.process(voice[:, a * B:b * B], sl[:, a * B:b * B], sr[:, a * B:b * B])
            outL.append(l); outR.append(r)
            for s in range(S):
                pf[s] += eng.pitch_frames(s)
    finally:
        eng.close()
    outL, outR = np.concatenate(outL, axis=1), np.concatenate(outR, axis=1)
    for s in range(S):
        one = vp.Engine(fs, B, 1, max(b - a for a, b in zip(cuts, cuts[1:])), params=vp.default_params(**per_cut[0][s]))
        try:
            l1, r1 = [], []
            for c, (a, b) in enumerate(zip(cuts, cuts[1:])):
                one.set_params(vp.default_params(**per_cut[c][s]))
                l, r = one.process(voice[s:s + 1, a * B:b * B], sl[s:s + 1, a * B:b * B], sr[s:s + 1, a * B:b * B])
                l1.append(l[0]); r1.append(r[0])
        finally:
            one.close()
        assert np.array_equal(outL[s], np.concatenate(l1)) and np.array_equal(outR[s], np.concatenate(r1)), s
        sched = [(a, refbind.default_params(**per_cut[c][s])) for c, a in enumerate(cuts[:-1]) if c > 0]
        r = ref_run(fs, B, voice[s], sl[s], sr[s], refbind.default_params(**per_cut[0][s]), schedule=sched)
        assert_audio(r["outL"], outL[s], "stream %d L" % s)
        assert_audio(r["outR"], outR[s], "stream %d R" % s)
        assert_decisions(compare_decisions(vp, oracle_decisions(r["pitch"]), pf[s]), "stream %d" % s)


@pytest.mark.gpu
def test_broadcast_getters_and_reset(vp):
    fs, S = 44100.0, 6
    n = int(fs * 3.0) // B * B
    voice, sl, sr = vp.synth_host(fs, S, n, flavour=0, first_stream=3200)
    P = dict(keyPitch=4, gainVoc=-3.0, gainPitch=-1.5, gainVoice=-30.0, gainSynth=-24.0)
    a = vp.Engine(fs, B, S, n // B, params=vp.default_params(**P))
    b = vp.Engine(fs, B, S, n // B)
    try:
        aL, aR = a.process(voice, sl, sr)
        b.set_stream_params(0, [vp.stream_params(**P)] * S)  # identical values for all streams == set_params
        bL, bR = b.process(voice, sl, sr)
        assert np.array_equal(aL, bL) and np.array_equal(aR, bR)
        # what was set is what the getter returns; reset keeps it
        items = spread(S)
        b.set_stream_params(0, items)
        want = [vp.stream_params(**it).as_dict() for it in items]
        assert b.stream_params() == want
        assert b.stream_params(2, 3) == want[2:5]
        b.reset()
        assert b.stream_params() == want
        # after the reset the streams restart with their own values: == a fresh batch with the same per-stream values
        rL, rR = b.process(voice, sl, sr)
        fresh = run_batch(vp, fs, B, voice, sl, sr, items)
        assert np.array_equal(rL, fresh["outL"]) and np.array_equal(rR, fresh["outR"])
        # a later set_params overwrites every stream's values
        b.set_params(vp.default_params(**P))
        assert b.stream_params() == [vp.stream_params(**P).as_dict()] * S
        b.reset()
        cL, cR = b.process(voice, sl, sr)
        assert np.array_equal(cL, aL) and np.array_equal(cR, aR)
    finally:
        a.close()
        b.close()


@pytest.mark.gpu
def test_streaming_per_stream_changes_need_no_capture(vp):
    """Per-stream key and gain changes between vp_engine_stream_block calls: block by block equal to vp_engine_process_host
    with the same changes, and no new graph capture after them."""
    fs, Bs, S, nb = 44100.0, 128, 5, 120
    voice, sl, _ = vp.synth_host(fs, S, nb * Bs, flavour=0, first_stream=3300)
    start = [dict(keyPitch=k, gainVoc=g) for k, g in zip((0, 3, 5, 9, 12), (0.0, -6.0, 2.0, -20.0, 6.0))]
    changes = {60: {1: dict(keyPitch=7), 3: dict(gainPitch=-12.0)}, 90: {0: dict(gainVoc=-9.0, keyPitch=11), 4: dict(keyPitch=2)}}
    ref = vp.Engine(fs, Bs, S, 1)
    eng = vp.Engine(fs, Bs, S, 1)
    try:
        for e in (ref, eng):
            e.set_stream_params(0, start)
        hv, hs, ho = eng.stream_buffers()
        captures = None
        for b in range(nb):
            for s, d in changes.get(b, {}).items():
                ref.set_stream_params(s, [d])
                eng.set_stream_params(s, [d])
            if b == 60:
                captures = eng.stream_stats()["graph_captures"]
            x = slice(b * Bs, (b + 1) * Bs)
            rl, _ = ref.process(voice[:, x], sl[:, x], None, want_right=False)
            hv[:] = voice[:, x]
            hs[:] = sl[:, x]
            eng.stream_block()
            assert np.array_equal(ho, rl), "block %d" % b
        st = eng.stream_stats()
        assert st["graph_launches"] == nb and st["graph_captures"] == captures
    finally:
        ref.close()
        eng.close()


@pytest.mark.gpu
def test_set_during_asynchronous_call_does_not_change_it(vp):
    """process_device without sync, then set_stream_params, then sync: the call computes with the values it was issued
    with; the next call uses the new ones."""
    fs, S = 48000.0, 8
    n = int(fs * 20.0) // B * B
    voice, sl, _ = vp.synth_host(fs, S, n, flavour=0, first_stream=3400, want_right=False)
    old = [dict(keyPitch=s % 13, gainVoc=-2.0 * s) for s in range(S)]
    new = [dict(keyPitch=(s + 6) % 13, gainVoc=6.0 - s, gainPitch=-20.0, gainVoice=-10.0) for s in range(S)]

    def device_run(first_items, second_items):
        eng = vp.Engine(fs, B, S, n // B)
        bufs = [eng.device_alloc(S * n * 4) for _ in range(4)]
        try:
            eng.h2d(bufs[0], voice)
            eng.h2d(bufs[1], sl)
            eng.set_stream_params(0, first_items)
            eng.process_device(n // B, bufs[0], bufs[1], None, bufs[2], None, n, sync=False)
            if second_items is not None:
                eng.set_stream_params(0, second_items)
            eng.sync()
            out = np.zeros((S, n), np.float32)
            eng.d2h(out, bufs[2])
            return out
        finally:
            for p in bufs:
                eng.device_free(p)
            eng.close()
    assert np.array_equal(device_run(old, new), device_run(old, None))
    assert not np.array_equal(device_run(new, None), device_run(old, None))


@pytest.mark.gpu
def test_defined_mode_five_keys_in_one_engine(vp, oracle):
    """The U6 input (802 Hz pulse train, above every note table) in five keys in one engine: each stream equals the
    oracle's defined mode in its key (the note LUT rows are built per mode)."""
    from test_defined_mode import u6_input
    fs = 44100.0
    v6, s6 = u6_input()
    keys = (0, 3, 5, 9, 12)
    S = len(keys)
    eng = vp.Engine(fs, B, S, len(v6) // B)
    try:
        eng.set_mode(vp.VP_MODE_DEFINED)
        eng.set_stream_params(0, [dict(keyPitch=k) for k in keys])
        outL, _ = eng.process(np.tile(v6, (S, 1)), np.tile(s6, (S, 1)), None, want_right=False)
        frames = [eng.pitch_frames(s) for s in range(S)]
    finally:
        eng.close()
    try:
        oracle.set_defined(True)
        for s, k in enumerate(keys):
            r = oracle.run(fs, B, v6, s6, params=refbind.default_params(keyPitch=k), log=True)
            assert r["ub"] == 0
            assert_audio(r["outL"], outL[s], "key %d" % k)
            assert not any(f.flags & vp.PF_UB for f in frames[s]), k
            assert_decisions(compare_decisions(vp, oracle_decisions(r["pitch"]), frames[s]), "key %d" % k)
    finally:
        oracle.set_defined(False)


@pytest.mark.gpu
def test_host_paths_with_one_stream_dry_sidechain(vp):
    """process_host and process_pcm16 with the dry side-chain on for one stream only: that stream's R channel is its own
    (== the stream run alone), every other stream has L == R."""
    fs, S = 44100.0, 5
    n = 40 * B
    voice, sl, sr = vp.synth_host(fs, S, n, flavour=0, first_stream=3500)
    items = [dict(keyPitch=s * 2) for s in range(S)]
    items[2]["gainSynth"] = -12.0
    items[3]["gainVoice"] = -20.0
    eng = vp.Engine(fs, B, S, n // B, workspace_bytes=64 << 20)
    q = lambda a: np.clip(np.rint(a * np.float32(32768.0)), -32768, 32767).astype(np.int16)
    try:
        eng.set_stream_params(0, items)
        oL, oR = eng.process(voice, sl, sr)
        for s in range(S):
            assert np.array_equal(oL[s], oR[s]) == (s != 2), s
            one = run_alone(vp, fs, B, voice[s], sl[s], sr[s], items[s])
            assert np.array_equal(one["outL"], oL[s]) and np.array_equal(one["outR"], oR[s]), s
        qv, ql, qr = q(voice), q(sl), q(sr)
        fv, fl, fr = (a.astype(np.float32) * np.float32(1.0 / 32768.0) for a in (qv, ql, qr))
        eng.reset()
        pL, pR = eng.process_pcm16(qv, ql, qr)
        eng.reset()
        rL, rR = eng.process(fv, fl, fr)
        assert np.array_equal(pL, q(rL)) and np.array_equal(pR, q(rR))
        for s in range(S):
            assert np.array_equal(pL[s], pR[s]) == (s != 2), s
    finally:
        eng.close()


@pytest.mark.gpu
def test_stream_params_errors(vp):
    S = 3
    eng = vp.Engine(44100.0, 128, S, 1)
    try:
        eng.set_stream_params(0, spread(S))
        before = eng.stream_params()
        for bad in (dict(keyPitch=13), dict(keyPitch=-1), dict(gainVoc=6.5), dict(gainPitch=-60.5), dict(gainVoice=float("nan")),
                    dict(gainSynth=100.0)):
            with pytest.raises(vp.EngineError) as ei:
                eng.set_stream_params(0, [dict(keyPitch=1), bad])  # the valid first entry does not go in either
            assert ei.value.code == vp.VP_E_RANGE, bad
            assert eng.stream_params() == before
        for first, count in ((-1, 1), (S - 1, 2), (S, 1)):
            with pytest.raises(vp.EngineError) as ei:
                eng.set_stream_params(first, [dict(keyPitch=1)] * count)
            assert ei.value.code == vp.VP_E_ARG
            with pytest.raises(vp.EngineError) as ei:
                eng.stream_params(first, count)
            assert ei.value.code == vp.VP_E_ARG
        assert eng.lib.vp_engine_set_stream_params(eng.h, 0, 1, None) == vp.VP_E_ARG
        assert eng.stream_params() == before
        # streaming carries side-chain channel 0 only: the dry side-chain on any one stream is refused
        eng.stream_buffers()
        eng.set_stream_params(1, [dict(gainSynth=-10.0)])
        with pytest.raises(vp.EngineError) as ei:
            eng.stream_block()
        assert ei.value.code == vp.VP_E_ARG
        eng.set_stream_params(1, [dict(gainSynth=-59.0)])
        eng.stream_block()
    finally:
        eng.close()
    # before prepare
    lib = vp.load_library()
    h = C.c_void_p()
    assert lib.vp_engine_create(C.byref(h), 0) == vp.VP_OK
    try:
        arr = (vp.StreamParams * 1)(vp.stream_params())
        assert lib.vp_engine_set_stream_params(h, 0, 1, arr) == vp.VP_E_STATE
        assert lib.vp_engine_get_stream_params(h, 0, 1, arr) == vp.VP_E_STATE
    finally:
        lib.vp_engine_destroy(h)


@pytest.mark.gpu
def test_wav_manifest_tokens_set_each_jobs_key_and_gains(vp, tmp_path):
    from test_wav import read_f32, write_f32
    from vocoderproject_b200 import build as bld
    bld.build()
    tool = bld.build_wavbatch()
    fs, K = 44100.0, 8
    lens = [70000, 52000]
    toks = ["key=3 gainVoc=-6", "key=7 gainVoc=2 gainPitch=-3"]
    per = [dict(keyPitch=3, gainVoc=-6.0, gainSynth=-20.0), dict(keyPitch=7, gainVoc=2.0, gainPitch=-3.0, gainSynth=-20.0)]
    v, l, r = vp.synth_host(fs, 2, max(lens), flavour=0, first_stream=3600)
    lines = []
    for s, n in enumerate(lens):
        pv, ps, po = [str(tmp_path / ("%s%d.wav" % (k, s))) for k in "vso"]
        write_f32(pv, fs, [v[s, :n]])
        write_f32(ps, fs, [l[s, :n], r[s, :n]])
        lines.append("%s %s %s %s" % (pv, ps, po, toks[s]))
    man = tmp_path / "m.txt"
    man.write_text("\n".join(lines) + "\n")
    out = subprocess.run([tool, str(man), "--block", str(B), "--blocks-per-call", str(K), "--key", "0", "--gain-synth", "-20"],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    lat = json.loads(out.stdout.strip().splitlines()[-1])["latency_samples"]
    m = K * B
    n = (max(lens) + lat + m - 1) // m * m
    V, L, R = (np.zeros((2, n), np.float32) for _ in range(3))
    for s, nl in enumerate(lens):
        V[s, :nl], L[s, :nl], R[s, :nl] = v[s, :nl], l[s, :nl], r[s, :nl]
    eng = vp.Engine(fs, B, 2, n // B)
    try:
        eng.set_stream_params(0, per)
        refL, refR = eng.process(V, L, R)
    finally:
        eng.close()
    for s, nl in enumerate(lens):
        fs_o, x = read_f32(str(tmp_path / ("o%d.wav" % s)))
        assert fs_o == 44100 and x.shape == (nl, 2)
        assert np.array_equal(x[:, 0], refL[s, lat:lat + nl]) and np.array_equal(x[:, 1], refR[s, lat:lat + nl])
    # a token the front-end does not know is an error, not ignored
    man.write_text(lines[0] + " gainFoo=1\n")
    bad = subprocess.run([tool, str(man)], capture_output=True, text=True)
    assert bad.returncode == 2 and "manifest tokens" in bad.stderr
