"""Per-stream pitch-corrector LPC order (vp_engine_set_stream_pitch_orders, vp_engine_reserve_pitch_order): each stream of a
batch has its own lpcPitch, taken when the stream starts (prepare, reset, or its reset_streams), as PitchProcess::prepare
reads it.

CPU: the names are in the ABI list, the argument codes that need no device, and the two premises on the C oracle: an lpcPitch
change inside a running stream changes nothing (the order is read in prepare only), and zeros for whole grid-aligned blocks
followed by X equal X from a fresh prepare, at every order. GPU: batches with lpcPitch spread over 2..15 and over 2..100
equal, bit for bit, each stream alone in an engine whose vp_params carry its order (several passes, the host, device and
PCM16 paths, with per-stream keys, gains and vocoder orders) and match the reference; a set on a running stream waits for
its start; reset_streams, reset and prepare start streams as documented; set_params leaves the values alone; errors change
nothing; a uniform call launches what it launched before; streaming matches the host path; the WAV manifest's lpcPitch=."""
import ctypes as C
import json
import subprocess

import numpy as np
import pytest

import refbind
from common import assert_decisions, compare_decisions, oracle_decisions
from test_stream_orders import keys_gains, reference_check, spread_orders
from test_stream_schedule import assert_audio, assert_same, collect, device_call, finish, new_res, ref_run


# ---------------------------------------------------------------------------------------------------------- CPU
def test_names_in_abi(vp):
    for name in ("vp_engine_reserve_pitch_order", "vp_engine_set_stream_pitch_orders", "vp_engine_get_stream_pitch_orders"):
        assert name in vp.ABI_SYMBOLS


def test_null_engine_and_arguments(vp):
    lib = vp.load_library()
    v = (C.c_int * 2)(9, 20)
    assert lib.vp_engine_reserve_pitch_order(None, 20) == vp.VP_E_ARG
    assert lib.vp_engine_set_stream_pitch_orders(None, 0, 2, v) == vp.VP_E_ARG
    assert lib.vp_engine_set_stream_pitch_orders(None, 0, 0, None) == vp.VP_E_ARG
    assert lib.vp_engine_get_stream_pitch_orders(None, 0, 2, v, None) == vp.VP_E_ARG
    assert lib.vp_engine_get_stream_pitch_orders(None, 0, 0, None, None) == vp.VP_E_ARG


@pytest.mark.parametrize("fs", [44100.0, 48000.0], ids=["44k1", "48k"])
def test_oracle_lpc_pitch_read_in_prepare_only(vp, oracle, fs):
    """lpcPitch changed by the automation of a running stream (at several blocks, to both ends of its range): output and
    pitch records bit-identical to the run without the change."""
    B, nb = 1024, 30
    voice, sl, sr = vp.synth_host(fs, 1, nb * B, flavour=0, first_stream=7000)
    base = refbind.default_params()
    r0 = oracle.run(fs, B, voice[0], sl[0], synthR=sr[0], params=base, log=True)
    sched = [(7, refbind.default_params(lpcPitch=2)), (13, refbind.default_params(lpcPitch=100)),
             (20, refbind.default_params(lpcPitch=31))]
    r1 = oracle.run(fs, B, voice[0], sl[0], synthR=sr[0], params=base, log=True, schedule=sched)
    assert np.array_equal(r0["outL"], r1["outL"]) and np.array_equal(r0["outR"], r1["outR"])
    assert [bytes(f) for f in r0["pitch"]] == [bytes(f) for f in r1["pitch"]]


@pytest.mark.parametrize("p", [2, 9, 15, 20, 100])
def test_oracle_zero_prefix_is_a_fresh_start(vp, oracle, p):
    """k grid-aligned blocks of zeros (every 3rd block at 44.1 kHz / 1024 is on both frame grids' prepare phase), then X, at
    order p: the output from block k on is bit-identical to X from a fresh prepare at order p. This is what a stream handed
    to a new instance with reset_streams at such a block is compared with."""
    fs, B, nb = 44100.0, 1024, 24
    voice, sl, sr = vp.synth_host(fs, 1, nb * B, flavour=0, first_stream=7100)
    prm = refbind.default_params(lpcPitch=p)
    fresh = oracle.run(fs, B, voice[0], sl[0], synthR=sr[0], params=prm)
    for k in (3, 6):
        z = np.zeros(k * B, np.float32)
        late = oracle.run(fs, B, np.concatenate([z, voice[0]]), np.concatenate([z, sl[0]]), synthR=np.concatenate([z, sr[0]]),
                          params=prm)
        assert np.array_equal(late["outL"][k * B:], fresh["outL"]), (p, k)
        assert np.array_equal(late["outR"][k * B:], fresh["outR"]), (p, k)


# ---------------------------------------------------------------------------------------------------------- GPU helpers
def pitch_spread(S, lo, hi):
    """lpcPitch lo .. hi spread over S streams (both ends included)."""
    return [int(x) for x in np.linspace(lo, hi, S).round()]


def quant16(a):
    return np.clip(np.rint(a * np.float32(32768.0)), -32768, 32767).astype(np.int16)


def call(eng, path, voice, sl, sr):
    if path == "pcm16":
        return eng.process_pcm16(quant16(voice), quant16(sl), quant16(sr))
    if path == "device":
        return device_call(eng, voice, sl, sr)
    return eng.process(voice, sl, sr)


def batch_run(vp, fs, B, voice, sl, sr, porders, sp=None, vorders=None, workspace_bytes=0, reserve=None, path="host"):
    S, n = voice.shape
    eng = vp.Engine(fs, B, S, n // B, workspace_bytes=workspace_bytes, reserve_pitch_order=reserve)
    res = new_res(S)
    try:
        if sp is not None:
            eng.set_stream_params(0, sp)
        if vorders is not None:
            eng.set_stream_orders(0, vorders)
        eng.set_stream_pitch_orders(0, porders)
        assert eng.stream_pitch_orders() == (list(porders), list(porders))
        l, r = call(eng, path, voice, sl, sr)
        collect(eng, S, res, l, r)
        res = finish(res)
        res["passes"] = -(-S // eng.info()["streams_per_pass"])
        res["pitch_orders"] = eng.stream_pitch_orders()
        return res
    finally:
        eng.close()


def solo_runs(vp, fs, B, voice, sl, sr, porders, sp=None, vorders=None, path="host", streams=None):
    """Each stream alone in an engine whose vp_params carry its lpcPitch (and its key, gains and vocoder orders)."""
    S, n = voice.shape
    streams = list(range(S)) if streams is None else streams
    res = new_res(S)
    outs = []
    for s in streams:
        kw = dict(lpcPitch=porders[s])
        if sp is not None:
            kw.update(sp[s])
        if vorders is not None:
            kw.update(lpcVoice=vorders[s][0], lpcSynth=vorders[s][1])
        eng = vp.Engine(fs, B, 1, n // B, params=vp.default_params(**kw))
        try:
            l, r = call(eng, path, voice[s:s + 1], sl[s:s + 1], sr[s:s + 1])
            outs.append((l[0], r[0]))
            res["pf"][s] += [bytes(f) for f in eng.pitch_frames(0)]
            res["frames"][s] += eng.pitch_frames(0)
            vf = eng.voc_frames(0)
            for k in vf:
                res["vf"][s][k].append(vf[k])
        finally:
            eng.close()
    res["outL"] = [np.stack([o[0] for o in outs])]
    res["outR"] = [np.stack([o[1] for o in outs])]
    return finish(res)


def assert_streams_same(solo, batch, streams, what):
    """solo holds the listed streams in order (solo_runs(..., streams=...)), batch all of them."""
    for k, s in enumerate(streams):
        assert np.array_equal(solo["outL"][k], batch["outL"][s]), "%s: stream %d outL" % (what, s)
        assert np.array_equal(solo["outR"][k], batch["outR"][s]), "%s: stream %d outR" % (what, s)
        assert solo["pf"][s] == batch["pf"][s], "%s: stream %d pitch frame records" % (what, s)


# ---------------------------------------------------------------------------------------------------------- GPU: spread <= 15
@pytest.fixture(scope="module", params=[(44100.0, 1024, 45), (48000.0, 1024, 45), (48000.0, 128, 300)],
                ids=["44k1-1024", "48k-1024", "48k-128"])
def low_case(request, vp):
    fs, B, nb = request.param
    S = 26
    voice, sl, sr = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=7200)
    porders = pitch_spread(S, 2, 15)
    one = batch_run(vp, fs, B, voice, sl, sr, porders)
    return dict(fs=fs, B=B, nb=nb, S=S, voice=voice, sl=sl, sr=sr, porders=porders, one=one)


@pytest.mark.gpu
def test_spread_to_15_equals_each_stream_alone(vp, low_case):
    c = low_case
    assert min(c["porders"]) == 2 and max(c["porders"]) == 15
    assert_same(solo_runs(vp, c["fs"], c["B"], c["voice"], c["sl"], c["sr"], c["porders"]), c["one"], c["S"],
                "lpcPitch 2..15 against solo engines")


@pytest.mark.gpu
def test_spread_to_15_matches_reference(vp, low_case):
    c = low_case
    if c["B"] == 128:
        pytest.skip("one block size is enough against the reference; the solo test covers B = 128 bit for bit")
    reference_check(vp, c["fs"], c["B"], c["voice"], c["sl"], c["sr"], c["one"],
                    lambda s: refbind.default_params(lpcPitch=c["porders"][s]))


@pytest.mark.gpu
def test_with_keys_gains_and_vocoder_orders(vp, low_case):
    """lpcPitch, key, gains, lpcVoice and lpcSynth all per stream: still each stream alone."""
    c = low_case
    if c["B"] == 128:
        pytest.skip("covered at B = 1024")
    S = c["S"]
    sp = keys_gains(S, seed=int(c["fs"]) + 1)
    vo = spread_orders(S)[::-1]
    args = (vp, c["fs"], c["B"], c["voice"], c["sl"], c["sr"], c["porders"])
    assert_same(solo_runs(*args, sp=sp, vorders=vo), batch_run(*args, sp=sp, vorders=vo), S, "all per-stream values")


# ---------------------------------------------------------------------------------------------------------- GPU: spread <= 100
@pytest.fixture(scope="module", params=[(44100.0, 1024, 45), (48000.0, 1024, 45)], ids=["44k1", "48k"])
def wide_case(request, vp):
    fs, B, nb = request.param
    S = 26
    voice, sl, sr = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=7300)
    porders = pitch_spread(S, 2, 100)
    one = batch_run(vp, fs, B, voice, sl, sr, porders, reserve=100)
    return dict(fs=fs, B=B, nb=nb, S=S, voice=voice, sl=sl, sr=sr, porders=porders, one=one)


@pytest.mark.gpu
def test_spread_to_100_equals_each_stream_alone(vp, wide_case):
    c = wide_case
    assert min(c["porders"]) == 2 and max(c["porders"]) == 100
    solo = solo_runs(vp, c["fs"], c["B"], c["voice"], c["sl"], c["sr"], c["porders"])
    assert_same(solo, c["one"], c["S"], "lpcPitch 2..100 against solo engines")


@pytest.mark.gpu
def test_spread_to_100_multi_pass_device_and_pcm16(vp, wide_case):
    c = wide_case
    fs, B, S, nb = c["fs"], c["B"], c["S"], c["nb"]
    args = (vp, fs, B, c["voice"], c["sl"], c["sr"], c["porders"])
    eng = vp.Engine(fs, B, S, nb, reserve_pitch_order=100)
    per = eng.info()["workspace_bytes"] // S
    eng.close()
    multi = batch_run(*args, workspace_bytes=7 * per + per // 2, reserve=100)
    assert multi["passes"] >= 3
    assert_same(c["one"], multi, S, "%d passes" % multi["passes"])
    assert_same(c["one"], batch_run(*args, reserve=100, path="device"), S, "device path")
    streams = [0, 5, 12, S - 1]
    assert_streams_same(solo_runs(*args, path="pcm16", streams=streams), batch_run(*args, reserve=100, path="pcm16"),
                        streams, "pcm16")


@pytest.mark.gpu
def test_spread_to_100_matches_reference(vp, wide_case):
    c = wide_case
    reference_check(vp, c["fs"], c["B"], c["voice"], c["sl"], c["sr"], c["one"],
                    lambda s: refbind.default_params(lpcPitch=c["porders"][s]))


@pytest.mark.gpu
def test_defined_mode_against_oracle(vp, oracle):
    """VP_MODE_DEFINED with four lpcPitch values in one batch on the U6 input: each stream equals the oracle's defined mode at
    its order."""
    from test_defined_mode import u6_input
    fs, B = 44100.0, 1024
    v6, s6 = u6_input()
    nb = len(v6) // B
    porders = [2, 15, 9, 40]
    S = len(porders)
    eng = vp.Engine(fs, B, S, nb, reserve_pitch_order=40)
    try:
        eng.set_mode(vp.VP_MODE_DEFINED)
        eng.set_stream_pitch_orders(0, porders)
        outL, _ = eng.process(np.tile(v6[:nb * B], (S, 1)), np.tile(s6[:nb * B], (S, 1)), None, want_right=False)
        frames = [eng.pitch_frames(s) for s in range(S)]
    finally:
        eng.close()
    try:
        oracle.set_defined(True)
        for s in range(S):
            r = oracle.run(fs, B, v6[:nb * B], s6[:nb * B], params=refbind.default_params(lpcPitch=porders[s]), log=True)
            assert_audio(r["outL"], outL[s], "stream %d" % s)
            assert_decisions(compare_decisions(vp, oracle_decisions(r["pitch"]), frames[s]), "stream %d" % s)
    finally:
        oracle.set_defined(False)


# ---------------------------------------------------------------------------------------------------------- GPU: starts
def run_steps(vp, fs, B, S, nb, voice, sl, sr, steps, reserve=32, init=None):
    """steps: (a, b) = process blocks a .. b in one call, or a callable(eng); returns (outL, outR, pitch orders, engine log)."""
    eng = vp.Engine(fs, B, S, nb, reserve_pitch_order=reserve)
    L, R, log = [], [], []
    try:
        if init is not None:
            eng.set_stream_pitch_orders(0, init)
        for st in steps:
            if callable(st):
                log.append(st(eng))
            else:
                a, b = st
                l, r = eng.process(voice[:, a * B:b * B], sl[:, a * B:b * B], sr[:, a * B:b * B])
                L.append(l); R.append(r)
        return np.concatenate(L, axis=1), np.concatenate(R, axis=1), eng.stream_pitch_orders(), log
    finally:
        eng.close()


@pytest.fixture(scope="module")
def start_case(vp):
    fs, B, S, nb = 44100.0, 1024, 6, 36
    voice, sl, sr = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=7400)
    init = [15, 4, 15, 11, 15, 15]
    plain = run_steps(vp, fs, B, S, nb, voice, sl, sr, [(0, nb)], init=init)
    return dict(fs=fs, B=B, S=S, nb=nb, voice=voice, sl=sl, sr=sr, init=init, plain=plain)


@pytest.mark.gpu
def test_set_on_running_stream_waits_for_its_start(vp, start_case):
    c = start_case
    fs, B, S, nb = c["fs"], c["B"], c["S"], c["nb"]
    args = (vp, fs, B, S, nb, c["voice"], c["sl"], c["sr"])
    got = run_steps(*args, [(0, 10), lambda e: e.set_stream_pitch_orders(2, [9, 24]), lambda e: e.stream_pitch_orders(),
                            (10, nb)], init=c["init"])
    assert np.array_equal(got[0], c["plain"][0]) and np.array_equal(got[1], c["plain"][1])
    inforce, nxt = got[3][1]
    assert inforce == c["init"] and nxt == [15, 4, 9, 24, 15, 15]
    assert got[2] == (c["init"], [15, 4, 9, 24, 15, 15])


@pytest.mark.gpu
@pytest.mark.parametrize("b", [15, 16, 17], ids=["aligned", "off1", "off2"])
def test_reset_streams_starts_with_the_new_order(vp, start_case, b):
    """Streams 2 and 3 get 9 and 24 while running and are reset at block b (15: on both grids' prepare phase; 16, 17: not):
    from b on each equals a solo engine at its new order fed zeros up to b and then the same input, bit for bit, and the
    reference on that input; every other stream is bit-identical to the run without the reset."""
    c = start_case
    fs, B, S, nb = c["fs"], c["B"], c["S"], c["nb"]
    voice, sl, sr = c["voice"], c["sl"], c["sr"]
    got = run_steps(vp, fs, B, S, nb, voice, sl, sr,
                    [(0, b), lambda e: e.set_stream_pitch_orders(2, [9, 24]), lambda e: e.reset_streams([2, 3]),
                     lambda e: e.stream_pitch_orders(), (b, nb)], init=c["init"])
    assert got[3][2] == ([15, 4, 9, 24, 15, 15], [15, 4, 9, 24, 15, 15])
    for s in (0, 1, 4, 5):
        assert np.array_equal(got[0][s], c["plain"][0][s]) and np.array_equal(got[1][s], c["plain"][1][s]), s
    for s, p in ((2, 9), (3, 24)):
        assert np.array_equal(got[0][s, :b * B], c["plain"][0][s, :b * B])
        x = [np.concatenate([np.zeros((1, b * B), np.float32), a[s:s + 1, b * B:]], axis=1) for a in (voice, sl, sr)]
        eng = vp.Engine(fs, B, 1, nb, params=vp.default_params(lpcPitch=p))
        try:
            l, r = eng.process(*x)
        finally:
            eng.close()
        assert np.array_equal(got[0][s, b * B:], l[0, b * B:]) and np.array_equal(got[1][s, b * B:], r[0, b * B:]), (s, b)
        ref = ref_run(fs, B, x[0][0], x[1][0], x[2][0], refbind.default_params(lpcPitch=p))
        assert_audio(ref["outL"][b * B:], got[0][s, b * B:], "stream %d after reset at %d L" % (s, b))
        assert_audio(ref["outR"][b * B:], got[1][s, b * B:], "stream %d after reset at %d R" % (s, b))


@pytest.mark.gpu
def test_reset_and_prepare_start_every_stream(vp, start_case):
    """vp_engine_reset starts every stream with its set value (equal to a fresh engine given those values); vp_engine_prepare
    returns every stream to vp_params.lpcPitch."""
    c = start_case
    fs, B, S, nb = c["fs"], c["B"], c["S"], c["nb"]
    voice, sl, sr = c["voice"], c["sl"], c["sr"]
    new = [20, 4, 2, 11, 15, 32]
    got = run_steps(vp, fs, B, S, nb, voice, sl, sr,
                    [(0, 10), lambda e: e.set_stream_pitch_orders(0, new), lambda e: e.reset(), (0, nb)], init=c["init"])
    assert got[2] == (new, new)
    fresh = run_steps(vp, fs, B, S, nb, voice, sl, sr, [(0, nb)], init=new)
    assert np.array_equal(got[0][:, 10 * B:], fresh[0]) and np.array_equal(got[1][:, 10 * B:], fresh[1])
    eng = vp.Engine(fs, B, S, nb, reserve_pitch_order=32)
    try:
        eng.set_stream_pitch_orders(0, new)
        eng.process(voice[:, :5 * B], sl[:, :5 * B], sr[:, :5 * B])
        assert eng.lib.vp_engine_prepare(eng.h, fs, B, S, nb, 0) == vp.VP_OK
        assert eng.stream_pitch_orders() == ([15] * S, [15] * S)
    finally:
        eng.close()


@pytest.mark.gpu
def test_set_params_leaves_stream_values_alone(vp, start_case):
    """set_params before every call (what the facade does per block), with another lpcPitch in it: the per-stream values in
    force and next are unchanged, and so is the output."""
    c = start_case
    fs, B, S, nb = c["fs"], c["B"], c["S"], c["nb"]
    P = vp.default_params(lpcPitch=30)
    steps = [(0, 6), lambda e: e.set_stream_pitch_orders(1, [7])]
    for a in range(6, nb, 6):
        steps += [lambda e: e.set_params(P), (a, a + 6)]
    got = run_steps(vp, fs, B, S, nb, c["voice"], c["sl"], c["sr"], steps, init=c["init"])
    assert np.array_equal(got[0], c["plain"][0]) and np.array_equal(got[1], c["plain"][1])
    assert got[2] == (c["init"], [15, 7, 15, 11, 15, 15])


@pytest.mark.gpu
def test_errors_change_nothing(vp, start_case):
    c = start_case
    fs, B, S, nb = c["fs"], c["B"], c["S"], c["nb"]
    lib = vp.load_library()
    h = C.c_void_p()
    assert lib.vp_engine_create(C.byref(h), 0) == vp.VP_OK
    try:
        v = (C.c_int * 1)(9)
        assert lib.vp_engine_set_stream_pitch_orders(h, 0, 1, v) == vp.VP_E_STATE
        assert lib.vp_engine_get_stream_pitch_orders(h, 0, 1, v, v) == vp.VP_E_STATE
        assert lib.vp_engine_reserve_pitch_order(h, 101) == vp.VP_E_RANGE
        assert lib.vp_engine_reserve_pitch_order(h, -1) == vp.VP_E_RANGE
    finally:
        lib.vp_engine_destroy(h)
    steps = [(0, 10)]
    codes = []

    def attempt(first, values, code):
        def f(e):
            before = e.stream_pitch_orders()
            with pytest.raises(vp.EngineError) as ei:
                e.set_stream_pitch_orders(first, values)
            assert e.stream_pitch_orders() == before
            codes.append((ei.value.code, code))
        return f
    for first, values, code in [(S - 1, [9, 9], vp.VP_E_ARG), (-1, [9], vp.VP_E_ARG), (0, [9, 1], vp.VP_E_RANGE),
                                (0, [9, 101], vp.VP_E_RANGE), (2, [9, 33], vp.VP_E_STATE)]:
        steps.append(attempt(first, values, code))

    def raw(e):
        before = e.stream_pitch_orders()
        assert e.lib.vp_engine_set_stream_pitch_orders(e.h, 0, 1, None) == vp.VP_E_ARG
        assert e.lib.vp_engine_set_stream_pitch_orders(e.h, 0, 0, None) == vp.VP_OK
        assert e.lib.vp_engine_get_stream_pitch_orders(e.h, S - 1, 2, None, None) == vp.VP_E_ARG
        assert e.lib.vp_engine_get_stream_pitch_orders(e.h, 0, S, None, None) == vp.VP_OK
        assert e.lib.vp_engine_reserve_pitch_order(e.h, 64) == vp.VP_E_STATE  # above the prepared size on a running engine
        assert e.stream_pitch_orders() == before
    steps += [raw, (10, nb)]
    got = run_steps(vp, fs, B, S, nb, c["voice"], c["sl"], c["sr"], steps, init=c["init"])
    assert all(a == b for a, b in codes) and len(codes) == 5, codes
    assert np.array_equal(got[0], c["plain"][0]) and np.array_equal(got[1], c["plain"][1])
    assert got[2] == (c["init"], c["init"])


# ---------------------------------------------------------------------------------------------------------- GPU: cost, streaming, WAV
@pytest.mark.gpu
def test_uniform_call_is_unchanged(vp):
    """All streams at 15 (set per stream) and all at 20 (set per stream within a reservation): the launches and bits of an
    engine whose vp_params carry that order and that never used the new calls. A reservation equal to vp_params.lpcPitch
    leaves the layout as it is; a larger one only widens the pitch rows."""
    fs, B, S, nb = 48000.0, 1024, 6, 30
    voice, sl, sr = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=7500)

    def run(params, porders, reserve=None):
        eng = vp.Engine(fs, B, S, nb, params=params, reserve_pitch_order=reserve)
        try:
            if porders is not None:
                eng.set_stream_pitch_orders(0, porders)
            k0 = eng.stats()["kernel_launches"]
            out = eng.process(voice, sl, sr)
            return eng.stats()["kernel_launches"] - k0, out, eng.info()
        finally:
            eng.close()
    k_plain, (l0, r0), info0 = run(vp.default_params(), None)
    k_set, (l1, r1), info1 = run(vp.default_params(), [15] * S)
    assert k_set == k_plain and np.array_equal(l0, l1) and np.array_equal(r0, r1) and info1 == info0
    assert run(vp.default_params(), None, reserve=15)[2] == info0
    k_plain, (l0, r0), _ = run(vp.default_params(lpcPitch=20), None)
    k_set, (l1, r1), info2 = run(vp.default_params(), [20] * S, reserve=20)
    assert k_set == k_plain and np.array_equal(l0, l1) and np.array_equal(r0, r1)
    assert info2["workspace_bytes"] >= info0["workspace_bytes"]


@pytest.mark.gpu
def test_streaming_matches_host_and_reset_costs_at_most_one_capture(vp):
    """stream_block over a mixed-order batch equals process_host block by block; a reset_streams that gives a stream a new
    order mid-stream (the batch stays mixed at the same widest order) matches the host path cut at that block and costs at
    most one capture more than the run without it."""
    fs, B, S, nb, b = 44100.0, 128, 8, 160, 61
    voice, sl, _ = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=7600, want_right=False)
    init = pitch_spread(S, 2, 15)

    def host(reset):
        eng = vp.Engine(fs, B, S, nb)
        try:
            eng.set_stream_pitch_orders(0, init)
            if not reset:
                return eng.process(voice, sl, None, want_right=False)[0]
            l0, _ = eng.process(voice[:, :b * B], sl[:, :b * B], None, want_right=False)
            eng.set_stream_pitch_orders(3, [12])
            eng.reset_streams([3])
            l1, _ = eng.process(voice[:, b * B:], sl[:, b * B:], None, want_right=False)
            return np.concatenate([l0, l1], axis=1)
        finally:
            eng.close()

    def stream(reset):
        eng = vp.Engine(fs, B, S, 1)
        out = np.zeros_like(voice)
        try:
            eng.set_stream_pitch_orders(0, init)
            hv, hs, ho = eng.stream_buffers()
            for k in range(nb):
                if reset and k == b:
                    eng.set_stream_pitch_orders(3, [12])
                    eng.reset_streams([3])
                hv[:] = voice[:, k * B:(k + 1) * B]
                hs[:] = sl[:, k * B:(k + 1) * B]
                eng.stream_block()
                out[:, k * B:(k + 1) * B] = ho
            return out, eng.stream_stats()["graph_captures"]
        finally:
            eng.close()
    plain, cap0 = stream(False)
    assert np.array_equal(plain, host(False))
    reset, cap1 = stream(True)
    assert np.array_equal(reset, host(True))
    assert not np.array_equal(reset[3], plain[3])
    assert cap1 - cap0 <= 1, (cap0, cap1)


@pytest.mark.gpu
def test_wav_manifest_pitch_tokens(vp, tmp_path):
    """lpcPitch= on manifest lines (one job above 15, reserved from the manifest): each job equals that job alone in an engine
    whose vp_params carry its order, through the facade that calls set_params before every block."""
    from test_wav import read_f32, write_f32
    from vocoderproject_b200 import build as b
    b.build()
    tool = b.build_wavbatch()
    fs, B, K, n = 44100.0, 1024, 8, 60000
    v, l, r = vp.synth_host(fs, 3, n, flavour=0, first_stream=7700)
    toks = ["lpcPitch=6", "", "lpcPitch=37 key=3"]
    params = [dict(lpcPitch=6), dict(), dict(lpcPitch=37, keyPitch=3)]
    lines = []
    for s in range(3):
        pv, ps, po = [str(tmp_path / ("%s%d.wav" % (k, s))) for k in "vso"]
        write_f32(pv, fs, [v[s]])
        write_f32(ps, fs, [l[s], r[s]])
        lines.append("%s %s %s %s" % (pv, ps, po, toks[s]))
    man = tmp_path / "m.txt"
    man.write_text("\n".join(lines) + "\n")
    out = subprocess.run([tool, str(man), "--block", str(B), "--blocks-per-call", str(K), "--keep-latency"],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert json.loads(out.stdout.strip().splitlines()[-1])["streams"] == 3
    m = -(-n // (K * B)) * K * B
    for s in range(3):
        _, x = read_f32(str(tmp_path / ("o%d.wav" % s)))
        pad = lambda a: np.concatenate([a[s:s + 1], np.zeros((1, m - n), np.float32)], axis=1)
        eng = vp.Engine(fs, B, 1, m // B, params=vp.default_params(**params[s]))
        try:
            sl_, sr_ = eng.process(pad(v), pad(l), pad(r))
        finally:
            eng.close()
        assert np.array_equal(x[:, 0], sl_[0, :n]) and np.array_equal(x[:, 1], sr_[0, :n]), "job %d" % s
