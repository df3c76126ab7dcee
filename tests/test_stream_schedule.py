"""Block-accurate per-stream automation (vp_stream_event, vp_engine_schedule_stream_params): a stream's key and gains change
at any block, also inside one process call.

CPU: the struct layout matches the header, the argument codes that need no device, and the premise on the C oracle: a
change at block b reaches the output exactly from the first read site in block b or later (the start of the first chunk
handled there for gainPitch, the first frame start for gainVoc / keyPitch, the block itself for the dry gains).
GPU: a pitch gain change between calls where a chunk straddles the cut matches the reference; one scheduled call equals, bit
for bit, the same schedule cut into calls at every event with vp_engine_set_stream_params between them and cut at random
blocks with the schedule queued up front (several passes, device / host / PCM16 paths); each stream matches the reference
run with its own schedule; streaming consumes events at their blocks; the interplay with reset, reset_streams,
set_stream_params, asynchronous calls and errors is as documented; a call without events in range launches nothing extra
and a scheduled call one kernel more."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import refbind
from common import MAXABS_MAX, SNR_MIN_DB, assert_decisions, compare_decisions, maxabs, oracle_decisions, snr_db

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("gainPitch", "gainVoice", "gainSynth", "gainVoc", "keyPitch")

LAYOUT_PROBE = r"""
#include <stddef.h>
#include <stdio.h>
#include "vp_engine.h"
int main(void) {
    printf("%zu %zu %zu %zu %zu %zu\n", sizeof(vp_stream_event), offsetof(vp_stream_event, stream),
           offsetof(vp_stream_event, reserved), offsetof(vp_stream_event, block), offsetof(vp_stream_event, p),
           offsetof(vp_stream_event, pad));
    return 0;
}
"""


# ---------------------------------------------------------------------------------------------------------- CPU
def test_stream_event_layout_matches_header(vp, tmp_path):
    E = vp.StreamEvent
    assert C.sizeof(E) == 40
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler to read the header's layout")
    src = tmp_path / "probe.c"
    src.write_text(LAYOUT_PROBE)
    exe = str(tmp_path / "probe")
    subprocess.check_call([cc, "-I", os.path.join(ROOT, "include"), "-o", exe, str(src)])
    got = [int(x) for x in subprocess.check_output([exe], text=True).split()]
    assert got == [C.sizeof(E), E.stream.offset, E.reserved.offset, E.block.offset, E.p.offset, E.pad.offset]
    assert "vp_engine_schedule_stream_params" in vp.ABI_SYMBOLS


def test_schedule_null_engine_is_an_argument_error(vp):
    lib = vp.load_library()
    arr = (vp.StreamEvent * 1)()
    assert lib.vp_engine_schedule_stream_params(None, arr, 1) == vp.VP_E_ARG
    assert lib.vp_engine_schedule_stream_params(None, None, 0) == vp.VP_E_ARG


def _first_diff(a, b):
    d = np.flatnonzero(a != b)
    return int(d[0]) if len(d) else None


def _ceil_to(x, m):
    return -(-x // m) * m


@pytest.mark.parametrize("fs,B,blocks", [(48000.0, 1024, (30, 31, 45)), (48000.0, 128, (240, 241)),
                                         (44100.0, 128, (240, 241)), (44100.0, 1024, (30, 31))],
                         ids=["48k-1024", "48k-128", "44k1-128", "44k1-1024"])
def test_oracle_pitch_gain_reaches_output_at_first_chunk_of_block(vp, oracle, fs, B, blocks):
    """A gainPitch change (-6 -> +3 dB) at block b changes nothing before the start of the first chunk handled in block b or
    later, and changes that chunk: chunks start at multiples of the chunk length c (pitchBool on throughout)."""
    c = oracle.sizes_for(fs, B)["chunk"]
    nb = max(blocks) + 20
    voice, sl, sr = vp.synth_host(fs, 1, nb * B, flavour=0, first_stream=4000)
    base = refbind.default_params(gainPitch=-6.0)
    r0 = oracle.run(fs, B, voice[0], sl[0], synthR=sr[0], params=base)
    for b in blocks:
        r1 = oracle.run(fs, B, voice[0], sl[0], synthR=sr[0], params=base,
                        schedule=[(b, refbind.default_params(gainPitch=3.0))])
        pos = _ceil_to(b * B, c)
        first = _first_diff(r0["outL"], r1["outL"])
        assert first is not None and pos <= first < pos + c, (b, pos - b * B, None if first is None else first - b * B)


@pytest.mark.parametrize("fs,B", [(48000.0, 1024), (44100.0, 128)], ids=["48k-1024", "44k1-128"])
def test_oracle_other_values_reach_output_at_their_read_site(vp, oracle, fs, B):
    """gainVoc (vocoder frame start), keyPitch (pitch frame start), gainVoice / gainSynth (the block) changed at block b:
    every sample before that read site is unchanged."""
    z = oracle.sizes_for(fs, B)
    nb = (60 if B == 1024 else 400)
    voice, sl, sr = vp.synth_host(fs, 1, nb * B, flavour=0, first_stream=4010)
    base = dict(keyPitch=12, gainVoc=-6.0, gainPitch=-3.0, gainVoice=-60.0, gainSynth=-60.0)
    r0 = oracle.run(fs, B, voice[0], sl[0], synthR=sr[0], params=refbind.default_params(**base))
    cases = [("gainVoc", 3.0, z["hopV"]), ("keyPitch", 3, z["hopP"]), ("gainVoice", -20.0, 1), ("gainSynth", -20.0, 1)]
    for b in ((nb // 2), (nb // 2) + 1):
        for field, val, grid in cases:
            new = dict(base)
            new[field] = val
            r1 = oracle.run(fs, B, voice[0], sl[0], synthR=sr[0], params=refbind.default_params(**base),
                            schedule=[(b, refbind.default_params(**new))])
            pos = _ceil_to(b * B, grid)
            first = _first_diff(r0["outL"], r1["outL"])
            assert first is not None and first >= pos, (field, b, pos, first)
            if grid == 1:
                assert first == pos, (field, b)


# ---------------------------------------------------------------------------------------------------------- GPU helpers
def assert_audio(ref, got, what):
    sn, mx = snr_db(ref, got), maxabs(ref, got)
    assert sn >= SNR_MIN_DB and mx <= MAXABS_MAX, "%s: SNR %.1f dB, max abs err %.3e" % (what, sn, mx)


def ref_run(fs, B, voice, sl, sr, params, schedule=None):
    """The reference's own C++ when it is built here, else the C oracle port (bit-identical to it)."""
    import oraclebind
    if refbind.available("strict"):
        return refbind.run(fs, B, voice, sl, synthR=sr, params=params, log=True, schedule=schedule)
    return oraclebind.run(fs, B, voice, sl, synthR=sr, params=params, log=True, schedule=schedule)


def random_values(rng, dry=True):
    v = dict(keyPitch=int(rng.integers(0, 13)), gainVoc=float(rng.choice([-18.0, -6.0, 0.0, 3.5])),
             gainPitch=float(rng.choice([-12.0, -6.0, 0.0, 3.0, 6.0])), gainVoice=-60.0, gainSynth=-60.0)
    if dry:
        v["gainVoice"] = float(rng.choice([-60.0, -59.0, -58.9, -20.0]))
        v["gainSynth"] = float(rng.choice([-60.0, -60.0, -24.0]))
    return v


def make_schedule(fs, B, S, nb, seed, dry=True):
    """Per stream: starting values and 3-8 events of all five fields at its own blocks, always including block 0, the last
    block and blocks where a pitch chunk straddles the block start."""
    rng = np.random.default_rng(seed)
    c = refbind_sizes(fs, B)["chunk"]
    straddle = [b for b in range(1, nb) if (b * B) % c != 0]
    base, events = [], []
    for s in range(S):
        base.append(random_values(rng, dry))
        k = int(rng.integers(3, 9))
        blocks = {0, nb - 1}
        if straddle:
            blocks.add(int(rng.choice(straddle)))
        while len(blocks) < k:
            blocks.add(int(rng.integers(1, nb)))
        for b in sorted(blocks):
            events.append((s, b, random_values(rng, dry)))
    return base, events


def refbind_sizes(fs, B):
    import oraclebind
    return oraclebind.sizes_for(fs, B)


def values_at(base, events, S, b):
    """[dict] the values of every stream in force at block b."""
    cur = [dict(x) for x in base]
    for s, eb, v in sorted(events, key=lambda e: e[1]):
        if eb <= b:
            cur[s] = dict(v)
    return cur


def collect(eng, S, res, outL, outR):
    res["outL"].append(outL)
    res["outR"].append(outR)
    for s in range(S):
        res["pf"][s] += [bytes(f) for f in eng.pitch_frames(s)]
        res["frames"][s] += eng.pitch_frames(s)
        vf = eng.voc_frames(s)
        for k in vf:
            res["vf"][s][k].append(vf[k])


def finish(res):
    out = dict(outL=np.concatenate(res["outL"], axis=1), outR=np.concatenate(res["outR"], axis=1), pf=res["pf"],
               frames=res["frames"])
    out["vf"] = [{k: np.concatenate(v[k]) if v[k] else np.zeros(0) for k in v} for v in res["vf"]]
    return out


def new_res(S):
    return dict(outL=[], outR=[], pf=[[] for _ in range(S)], frames=[[] for _ in range(S)],
                vf=[{k: [] for k in ("gated", "EeVoice", "EeSynth", "g")} for _ in range(S)])


def run_cuts(vp, fs, B, voice, sl, sr, base, events, cuts, mode, workspace_bytes=0, path="host"):
    """mode "schedule": the whole schedule queued before the first call; "set": vp_engine_set_stream_params at every cut
    with the values in force there (the cuts must include every event block)."""
    S, n = voice.shape
    nb = n // B
    eng = vp.Engine(fs, B, S, nb, workspace_bytes=workspace_bytes)
    res = new_res(S)
    try:
        eng.set_stream_params(0, base)
        if mode == "schedule":
            eng.schedule_stream_params(events)
        for a, b in zip(cuts, cuts[1:]):
            if mode == "set":
                now = values_at(base, events, S, a)
                eng.set_stream_params(0, now)
            x = slice(a * B, b * B)
            if path == "host":
                l, r = eng.process(voice[:, x], sl[:, x], sr[:, x])
            elif path == "pcm16":
                l, r = eng.process_pcm16(voice[:, x], sl[:, x], sr[:, x])
            else:
                l, r = device_call(eng, voice[:, x], sl[:, x], sr[:, x])
            collect(eng, S, res, l, r)
        res = finish(res)
        res["passes"] = -(-S // eng.info()["streams_per_pass"])
        res["stream_params"] = eng.stream_params()
        return res
    finally:
        eng.close()


def device_call(eng, voice, sl, sr):
    S, n = voice.shape
    bufs = [eng.device_alloc(S * n * 4) for _ in range(5)]
    try:
        eng.h2d(bufs[0], np.ascontiguousarray(voice))
        eng.h2d(bufs[1], np.ascontiguousarray(sl))
        eng.h2d(bufs[2], np.ascontiguousarray(sr))
        eng.process_device(n // eng.block, bufs[0], bufs[1], bufs[2], bufs[3], bufs[4], n)
        l, r = np.zeros((S, n), np.float32), np.zeros((S, n), np.float32)
        eng.d2h(l, bufs[3])
        eng.d2h(r, bufs[4])
        return l, r
    finally:
        for p in bufs:
            eng.device_free(p)


def assert_same(a, b, S, what):
    for s in range(S):
        assert np.array_equal(a["outL"][s], b["outL"][s]), "%s: stream %d outL" % (what, s)
        assert np.array_equal(a["outR"][s], b["outR"][s]), "%s: stream %d outR" % (what, s)
        assert a["pf"][s] == b["pf"][s], "%s: stream %d pitch frame records" % (what, s)
        for k in ("gated", "EeVoice", "EeSynth", "g"):
            assert np.array_equal(a["vf"][s][k], b["vf"][s][k]), "%s: stream %d vocoder frames %s" % (what, s, k)


# ---------------------------------------------------------------------------------------------------------- GPU tests
@pytest.mark.gpu
@pytest.mark.parametrize("fs,B,blocks", [(48000.0, 1024, (30, 31, 45)), (44100.0, 128, (240, 241))], ids=["48k-1024", "44k1-128"])
def test_pitch_gain_change_between_calls_straddling_chunk(vp, fs, B, blocks):
    """gainPitch -6 -> +3 -> -6 ... dB changed between calls at blocks where a pitch chunk straddles the cut (48 kHz / 1024:
    calls cut there; 44.1 kHz / 128: streaming, one block per call): the output matches the reference with the same
    schedule. The chunk that straddles the cut keeps the gain of the block that handled it, also for its part after the cut."""
    nb = max(blocks) + 30
    voice, sl, _ = vp.synth_host(fs, 1, nb * B, flavour=0, first_stream=4100, want_right=False)
    gains = {b: (3.0 if k % 2 == 0 else -6.0) for k, b in enumerate(blocks)}
    sched = [(b, refbind.default_params(gainPitch=g)) for b, g in sorted(gains.items())]
    r = ref_run(fs, B, voice[0], sl[0], None, refbind.default_params(gainPitch=-6.0), schedule=sched)
    if B == 1024:
        cuts = [0] + sorted(blocks) + [nb]
        eng = vp.Engine(fs, B, 1, nb)
        out = []
        try:
            eng.set_stream_params(0, [dict(gainPitch=-6.0)])
            for a, b in zip(cuts, cuts[1:]):
                if a in gains:
                    eng.set_stream_params(0, [dict(gainPitch=gains[a])])
                l, _ = eng.process(voice[:, a * B:b * B], sl[:, a * B:b * B], None, want_right=False)
                out.append(l[0])
        finally:
            eng.close()
        out = np.concatenate(out)
    else:
        eng = vp.Engine(fs, B, 1, 1)
        out = np.zeros(nb * B, np.float32)
        try:
            eng.set_stream_params(0, [dict(gainPitch=-6.0)])
            hv, hs, ho = eng.stream_buffers()
            for b in range(nb):
                if b in gains:
                    eng.set_stream_params(0, [dict(gainPitch=gains[b])])
                hv[:] = voice[:, b * B:(b + 1) * B]
                hs[:] = sl[:, b * B:(b + 1) * B]
                eng.stream_block()
                out[b * B:(b + 1) * B] = ho[0]
        finally:
            eng.close()
    assert_audio(r["outL"], out, "gainPitch changed between calls at %r" % (blocks,))


CUT_CASES = [(44100.0, 1024, 90), (48000.0, 1024, 90), (48000.0, 128, 360), (44100.0, 1000, 90)]


@pytest.fixture(scope="module", params=CUT_CASES, ids=["44k1-1024", "48k-1024", "48k-128", "44k1-1000"])
def sched_case(request, vp):
    fs, B, nb = request.param
    S = 26
    voice, sl, sr = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=4200)
    base, events = make_schedule(fs, B, S, nb, seed=int(fs) + B)
    one = run_cuts(vp, fs, B, voice, sl, sr, base, events, [0, nb], "schedule")
    return dict(fs=fs, B=B, nb=nb, S=S, voice=voice, sl=sl, sr=sr, base=base, events=events, one=one)


@pytest.mark.gpu
def test_one_call_equals_any_cut(vp, sched_case):
    c = sched_case
    fs, B, nb, S = c["fs"], c["B"], c["nb"], c["S"]
    args = (vp, fs, B, c["voice"], c["sl"], c["sr"], c["base"], c["events"])
    one = c["one"]
    ev_cuts = sorted({0, nb} | {b for _, b, _ in c["events"]})
    assert_same(one, run_cuts(*args, ev_cuts, "set"), S, "cut at every event with set_stream_params")
    rng = np.random.default_rng(7)
    rnd = sorted({0, nb} | set(int(x) for x in rng.integers(1, nb, 6)))
    assert_same(one, run_cuts(*args, rnd, "schedule"), S, "cut at %r, schedule up front" % rnd)
    # the host's values afterwards: those in force at the last block
    assert one["stream_params"] == [vp.stream_params(**v).as_dict() for v in values_at(c["base"], c["events"], S, nb - 1)]


@pytest.mark.gpu
def test_one_call_equals_any_cut_multi_pass_and_paths(vp, sched_case):
    """The same with a workspace that forces >= 3 passes (the block table is read at streamBase + stream of the pass), and on
    the device and PCM16 paths."""
    c = sched_case
    if c["B"] == 1000:
        pytest.skip("one block size is enough for the pass / path variants")
    fs, B, nb, S = c["fs"], c["B"], c["nb"], c["S"]
    args = (vp, fs, B, c["voice"], c["sl"], c["sr"], c["base"], c["events"])
    eng = vp.Engine(fs, B, S, nb)
    per = eng.info()["workspace_bytes"] // S
    eng.close()
    ws = 7 * per + per // 2
    ev_cuts = sorted({0, nb} | {b for _, b, _ in c["events"]})
    multi = run_cuts(*args, [0, nb], "schedule", workspace_bytes=ws)
    assert multi["passes"] >= 3
    assert_same(c["one"], multi, S, "%d passes" % multi["passes"])
    assert_same(c["one"], run_cuts(*args, ev_cuts, "set", workspace_bytes=ws), S, "cut at every event, several passes")
    assert_same(c["one"], run_cuts(*args, [0, nb], "schedule", path="device"), S, "device path")
    q = lambda a: np.clip(np.rint(a * np.float32(32768.0)), -32768, 32767).astype(np.int16)
    qargs = (vp, fs, B, q(c["voice"]), q(c["sl"]), q(c["sr"]), c["base"], c["events"])
    p1 = run_cuts(*qargs, [0, nb], "schedule", path="pcm16")
    p2 = run_cuts(*qargs, ev_cuts, "set", path="pcm16")
    assert np.array_equal(p1["outL"], p2["outL"]) and np.array_equal(p1["outR"], p2["outR"])


@pytest.mark.gpu
def test_scheduled_call_matches_reference_per_stream(vp, sched_case):
    from common import reference_runs  # noqa: F401  (same threads-over-streams pattern, with schedules)
    from concurrent.futures import ThreadPoolExecutor
    c = sched_case
    if c["B"] == 1000:
        pytest.skip("covered by the bit-exact cut tests")
    fs, B, nb, S = c["fs"], c["B"], c["nb"], c["S"]

    def one(s):
        sched = [(b, refbind.default_params(**v)) for t, b, v in c["events"] if t == s and b > 0]
        first = [v for t, b, v in c["events"] if t == s and b == 0]
        start = first[0] if first else c["base"][s]
        return ref_run(fs, B, c["voice"][s], c["sl"][s], c["sr"][s], refbind.default_params(**start), schedule=sched)
    with ThreadPoolExecutor(max_workers=max(1, len(os.sched_getaffinity(0)))) as ex:
        refs = list(ex.map(one, range(S)))
    res = c["one"]
    for s in range(S):
        what = "stream %d" % s
        assert_audio(refs[s]["outL"], res["outL"][s], what + " L")
        assert_audio(refs[s]["outR"], res["outR"][s], what + " R")
        assert_decisions(compare_decisions(vp, oracle_decisions(refs[s]["pitch"]), res["frames"][s]), what)


@pytest.mark.gpu
def test_defined_mode_five_keys_scheduled(vp, oracle):
    """The U6 input in defined mode, each stream moving through five keys at its own blocks in one call: equals the oracle's
    defined mode with the same schedule."""
    from test_defined_mode import u6_input
    fs, B = 44100.0, 1024
    v6, s6 = u6_input()
    nb = len(v6) // B
    keys = (0, 3, 5, 9, 12)
    S = 3
    events = []
    for s in range(S):
        for k, key in enumerate(keys[1:]):
            events.append((s, 1 + s + k * (nb // 5), dict(keyPitch=key)))
    eng = vp.Engine(fs, B, S, nb)
    try:
        eng.set_mode(vp.VP_MODE_DEFINED)
        eng.set_stream_params(0, [dict(keyPitch=keys[0])] * S)
        eng.schedule_stream_params(events)
        outL, _ = eng.process(np.tile(v6[:nb * B], (S, 1)), np.tile(s6[:nb * B], (S, 1)), None, want_right=False)
        frames = [eng.pitch_frames(s) for s in range(S)]
    finally:
        eng.close()
    try:
        oracle.set_defined(True)
        for s in range(S):
            sched = [(b, refbind.default_params(keyPitch=v["keyPitch"])) for t, b, v in events if t == s]
            r = oracle.run(fs, B, v6[:nb * B], s6[:nb * B], params=refbind.default_params(keyPitch=keys[0]), log=True,
                           schedule=sched)
            assert_audio(r["outL"], outL[s], "stream %d" % s)
            assert_decisions(compare_decisions(vp, oracle_decisions(r["pitch"]), frames[s]), "stream %d" % s)
    finally:
        oracle.set_defined(False)


def stream_run(vp, fs, B, voice, sl, base, events, via):
    """Streaming block by block; via = "schedule" (queued up front) or "set" (set_stream_params at each event block)."""
    S, n = voice.shape
    nb = n // B
    eng = vp.Engine(fs, B, S, 1)
    out = np.zeros((S, n), np.float32)
    try:
        eng.set_stream_params(0, base)
        if via == "schedule":
            eng.schedule_stream_params(events)
        hv, hs, ho = eng.stream_buffers()
        by = {}
        for s, b, v in events:
            by.setdefault(b, []).append((s, v))
        for b in range(nb):
            if via == "set":
                for s, v in by.get(b, []):
                    eng.set_stream_params(s, [v])
            hv[:] = voice[:, b * B:(b + 1) * B]
            hs[:] = sl[:, b * B:(b + 1) * B]
            eng.stream_block()
            out[:, b * B:(b + 1) * B] = ho
        return out, eng.stream_stats()
    finally:
        eng.close()


@pytest.mark.gpu
def test_streaming_consumes_events_at_their_blocks(vp):
    fs, B, S, nb = 44100.0, 128, 6, 200
    voice, sl, _ = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=4300, want_right=False)
    rng = np.random.default_rng(11)
    base = [random_values(rng, dry=False) for _ in range(S)]
    events = [(s, int(b), random_values(rng, dry=False)) for s in range(S) for b in rng.choice(np.arange(1, nb), 5, replace=False)]
    # == one process call with the same schedule, bit for bit
    eng = vp.Engine(fs, B, S, nb)
    try:
        eng.set_stream_params(0, base)
        eng.schedule_stream_params(events)
        ref, _ = eng.process(voice, sl, None, want_right=False)
    finally:
        eng.close()
    got, st = stream_run(vp, fs, B, voice, sl, base, events, "schedule")
    assert np.array_equal(got, ref)
    # key and gain events: no capture beyond what the block phases need
    _, st0 = stream_run(vp, fs, B, voice, sl, base, [], "schedule")
    assert st["graph_captures"] == st0["graph_captures"] and st["graph_launches"] == nb
    # a dry-voice event recaptures exactly as set_stream_params does
    dry = events + [(2, 50, dict(base[2], gainVoice=-20.0)), (2, 120, dict(base[2], gainVoice=-60.0))]
    a, sa = stream_run(vp, fs, B, voice, sl, base, dry, "schedule")
    b, sb = stream_run(vp, fs, B, voice, sl, base, dry, "set")
    assert np.array_equal(a, b)
    assert sa["graph_captures"] == sb["graph_captures"] > st0["graph_captures"]


def _engine_run(vp, fs, B, voice, sl, sr, base, steps, nbmax):
    """steps: list of callables (eng) -> None or (a, b) block ranges to process; returns concatenated outputs."""
    S = voice.shape[0]
    eng = vp.Engine(fs, B, S, nbmax)
    L, R = [], []
    try:
        eng.set_stream_params(0, base)
        for st in steps:
            if callable(st):
                st(eng)
            else:
                a, b = st
                l, r = eng.process(voice[:, a * B:b * B], sl[:, a * B:b * B], sr[:, a * B:b * B])
                L.append(l); R.append(r)
        return np.concatenate(L, axis=1), np.concatenate(R, axis=1)
    finally:
        eng.close()


@pytest.mark.gpu
def test_interplay_with_resets_and_set(vp):
    fs, B, S, nb = 44100.0, 1024, 5, 60
    voice, sl, sr = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=4400)
    rng = np.random.default_rng(5)
    base = [random_values(rng) for _ in range(S)]
    ev = [(s, int(b), random_values(rng)) for s in range(S) for b in (25 + s, 33 + 2 * s, 47)]
    drop1 = [e for e in ev if e[0] != 1]
    sched = lambda evs: (lambda eng: eng.schedule_stream_params(evs))
    # reset_streams drops the listed streams' pending events and keeps the others'
    a = _engine_run(vp, fs, B, voice, sl, sr, base, [sched(ev), (0, 20), lambda e: e.reset_streams([1]), (20, nb)], nb)
    b = _engine_run(vp, fs, B, voice, sl, sr, base, [sched(drop1), (0, 20), lambda e: e.reset_streams([1]), (20, nb)], nb)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    # reset drops every pending event
    a = _engine_run(vp, fs, B, voice, sl, sr, base, [(0, 10), sched([(s, b + 10, v) for s, b, v in ev]), lambda e: e.reset(), (0, 40)], nb)
    b = _engine_run(vp, fs, B, voice, sl, sr, base, [(0, 10), lambda e: e.reset(), (0, 40)], nb)
    assert np.array_equal(a[0][:, 10 * B:], b[0][:, 10 * B:]) and np.array_equal(a[1][:, 10 * B:], b[1][:, 10 * B:])
    # set_stream_params between calls with events pending: from the next block on, until the stream's next event
    X = dict(keyPitch=4, gainVoc=-3.0, gainPitch=2.0, gainVoice=-30.0, gainSynth=-60.0)
    a = _engine_run(vp, fs, B, voice, sl, sr, base, [sched(ev), (0, 20), lambda e: e.set_stream_params(3, [X]), (20, nb)], nb)
    cuts = sorted({20, nb} | {b for _, b, _ in ev})
    steps = [(0, 20)]
    state = [dict(x) for x in base]
    state[3] = dict(X)
    for lo, hi in zip(cuts, cuts[1:]):
        for s, b, v in ev:
            if b == lo:
                state[s] = dict(v)
        steps += [(lambda st: (lambda eng: eng.set_stream_params(0, st)))([dict(x) for x in state]), (lo, hi)]
    b = _engine_run(vp, fs, B, voice, sl, sr, base, steps, nb)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


@pytest.mark.gpu
def test_asynchronous_call_and_errors_queue_nothing(vp):
    fs, B, S = 48000.0, 1024, 6
    nb = 200
    voice, sl, _ = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=4500, want_right=False)
    n = nb * B
    later = [(s, nb + 3 + s, dict(keyPitch=(s + 5) % 13, gainVoc=-12.0, gainPitch=4.0)) for s in range(S)]

    def device_run(during):
        eng = vp.Engine(fs, B, S, nb)
        bufs = [eng.device_alloc(S * n * 4) for _ in range(3)]
        try:
            eng.h2d(bufs[0], voice)
            eng.h2d(bufs[1], sl)
            eng.process_device(nb, bufs[0], bufs[1], None, bufs[2], None, n, sync=False)
            if during:
                eng.schedule_stream_params(later)  # blocks after the running call
                with pytest.raises(vp.EngineError) as ei:  # a block of the running call has been issued
                    eng.schedule_stream_params([(0, nb - 1, dict(keyPitch=1))])
                assert ei.value.code == vp.VP_E_ARG
            eng.sync()
            out = np.zeros((S, n), np.float32)
            eng.d2h(out, bufs[2])
            return out
        finally:
            for p in bufs:
                eng.device_free(p)
            eng.close()
    assert np.array_equal(device_run(True), device_run(False))
    # error codes: nothing of a refused list is queued
    eng = vp.Engine(fs, B, S, 20)
    try:
        good = (0, 5, dict(keyPitch=3, gainVoc=-20.0))
        bad_range = [good, (1, 6, dict(gainVoc=6.5))]
        bad_args = [[good, (S, 6, dict())], [good, (-1, 6, dict())], [good, (0, -1, dict())]]
        with pytest.raises(vp.EngineError) as ei:
            eng.schedule_stream_params(bad_range)
        assert ei.value.code == vp.VP_E_RANGE
        for bad in bad_args:
            with pytest.raises(vp.EngineError) as ei:
                eng.schedule_stream_params(bad)
            assert ei.value.code == vp.VP_E_ARG
        lib = eng.lib
        assert lib.vp_engine_schedule_stream_params(eng.h, None, 1) == vp.VP_E_ARG
        assert lib.vp_engine_schedule_stream_params(eng.h, (vp.StreamEvent * 1)(), -1) == vp.VP_E_ARG
        assert lib.vp_engine_schedule_stream_params(eng.h, None, 0) == vp.VP_OK
        l1, _ = eng.process(voice[:, :20 * B], sl[:, :20 * B], None, want_right=False)
    finally:
        eng.close()
    eng = vp.Engine(fs, B, S, 20)
    try:
        l0, _ = eng.process(voice[:, :20 * B], sl[:, :20 * B], None, want_right=False)
    finally:
        eng.close()
    assert np.array_equal(l1, l0)
    # before prepare
    lib = vp.load_library()
    h = C.c_void_p()
    assert lib.vp_engine_create(C.byref(h), 0) == vp.VP_OK
    try:
        assert lib.vp_engine_schedule_stream_params(h, (vp.StreamEvent * 1)(), 1) == vp.VP_E_STATE
    finally:
        lib.vp_engine_destroy(h)


@pytest.mark.gpu
def test_launch_cost(vp):
    """A call with no event inside its blocks launches what a call of an engine that never scheduled anything launches; a
    call with events after its first block one kernel more (the table expansion). Same (stream, block) twice: the later
    one wins."""
    fs, B, S, nb = 44100.0, 1024, 4, 30
    voice, sl, sr = vp.synth_host(fs, S, 2 * nb * B, flavour=0, first_stream=4600)
    X = dict(keyPitch=7, gainVoc=-9.0, gainPitch=-3.0)

    def launches(steps):
        eng = vp.Engine(fs, B, S, nb)
        try:
            per = []
            for st in steps:
                if callable(st):
                    st(eng)
                    continue
                a, b = st
                k0 = eng.stats()["kernel_launches"]
                l, r = eng.process(voice[:, a * B:b * B], sl[:, a * B:b * B], sr[:, a * B:b * B])
                per.append((eng.stats()["kernel_launches"] - k0, l, r))
            return per
        finally:
            eng.close()
    plain = launches([(0, nb), (nb, 2 * nb)])
    # events beyond the first call and at the second call's first block only: no extra launch in either call
    edge = launches([lambda e: e.schedule_stream_params([(1, nb, X)]), (0, nb), (nb, 2 * nb)])
    assert [p[0] for p in edge] == [p[0] for p in plain]
    # events inside the second call: one more launch there
    inside = launches([lambda e: e.schedule_stream_params([(1, nb + 5, dict(X, keyPitch=2)), (1, nb + 5, X)]), (0, nb), (nb, 2 * nb)])
    assert inside[0][0] == plain[0][0] and inside[1][0] == plain[1][0] + 1
    # the later of two events for the same (stream, block) won: == set at a cut there
    cut = launches([(0, nb), (nb, nb + 5), lambda e: e.set_stream_params(1, [X]), (nb + 5, 2 * nb)])
    got = np.concatenate([inside[1][1]], axis=1)
    want = np.concatenate([cut[1][1], cut[2][1]], axis=1)
    assert np.array_equal(got, want)
