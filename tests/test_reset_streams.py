"""Per-stream reset (vp_engine_reset_streams): one stream of a running batch is handed to a new plug-in instance.

A reset stream continues as a stream that has received zeros on every input since prepare, with its own key and gains.
CPU: the argument codes without an engine, and the premise on the C oracle (zeros for a grid-aligned number of blocks
followed by X is X from a fresh prepare, bit for bit).
GPU: a reset stream equals, bit for bit, a twin that got zeros instead of the old user's audio (several grid phases, several
passes, bypass and order changes, defined mode, every process path, streaming); the other streams are untouched; the
reset stream matches the reference run on a zero prefix; at grid-aligned blocks it is a freshly prepared instance; the
asynchronous, cost and error semantics of the header hold."""
import ctypes as C

import numpy as np
import pytest

import refbind
from common import MAXABS_MAX, SNR_MIN_DB, assert_decisions, compare_decisions, maxabs, oracle_decisions, snr_db

DRY = dict(keyPitch=4, gainVoice=-12.0, gainSynth=-20.0)  # dry voice and dry side-chain on, a non-chromatic key


# ---------------------------------------------------------------------------------------------------------- CPU
def test_reset_streams_argument_codes_without_engine(vp):
    lib = vp.load_library()
    arr = (C.c_int * 1)(0)
    assert lib.vp_engine_reset_streams(None, arr, 1) == vp.VP_E_ARG
    assert lib.vp_engine_reset_streams(None, None, 1) == vp.VP_E_ARG
    assert lib.vp_engine_reset_streams(None, arr, -1) == vp.VP_E_ARG


@pytest.mark.parametrize("fs,B,k", [(44100.0, 1024, 3), (44100.0, 1024, 6), (44100.0, 128, 6)])
def test_oracle_silence_then_x_equals_fresh_x(vp, oracle, fs, B, k):
    """The state a reset writes is a fixed point of silence: zeros for k blocks (k * B a multiple of both frame hops)
    followed by X give, from block k on, exactly what X gives from a fresh prepare -- audio and every pitch decision."""
    n = int(fs * 2.0) // B * B
    v, l, r = vp.synth_host(fs, 1, n, flavour=0, first_stream=4000)
    z = np.zeros(k * B, np.float32)
    prm = refbind.default_params(**DRY)
    fresh = oracle.run(fs, B, v[0], l[0], synthR=r[0], params=prm, log=True)
    late = oracle.run(fs, B, np.concatenate([z, v[0]]), np.concatenate([z, l[0]]), synthR=np.concatenate([z, r[0]]),
                      params=prm, log=True)
    assert np.abs(fresh["outL"]).max() > 0.01 and not np.array_equal(fresh["outL"], fresh["outR"])
    assert np.array_equal(late["outL"][k * B:], fresh["outL"]) and np.array_equal(late["outR"][k * B:], fresh["outR"])
    pre = k * B // fresh["sizes"]["hopP"]
    assert k * B % fresh["sizes"]["hopP"] == 0 and k * B % fresh["sizes"]["hopV"] == 0
    assert oracle_decisions(late["pitch"])[pre:] == oracle_decisions(fresh["pitch"])


# ---------------------------------------------------------------------------------------------------------- GPU helpers
def quant(a):
    return np.clip(np.rint(a * np.float32(32768.0)), -32768, 32767).astype(np.int16)


def items_for(P):
    """P pairs of per-stream values (stream s and its twin s + P get the same): keys, gains, dry voice, dry side-chain."""
    base = []
    for s in range(P):
        it = dict(keyPitch=(3 * s + 1) % 13, gainVoc=-3.0 * (s % 4), gainPitch=2.0 - s, gainVoice=-60.0, gainSynth=-60.0)
        if s % 3 == 0:
            it["gainVoice"] = -14.0
        if s % 4 == 1:
            it["gainSynth"] = -18.0
        base.append(it)
    return base + [dict(it) for it in base]


def twin_inputs(vp, fs, B, P, calls, reset_call, first=4100, want_right=True):
    """Streams s < P: audio Y of an old user until their reset call, then X_s; their twins s + P: zeros, then the same X_s.
    reset_call[s] = the call before which stream s is reset."""
    starts = np.concatenate([[0], np.cumsum(calls)]) * B
    n = int(starts[-1])
    yv, yl, yr = vp.synth_host(fs, P, n, flavour=0, first_stream=first)
    xv, xl, xr = vp.synth_host(fs, P, n, flavour=2, first_stream=first + 50)
    V, L, R = (np.zeros((2 * P, n), np.float32) for _ in range(3))
    for s in range(P):
        a = int(starts[reset_call[s]])
        for D, y, x in ((V, yv, xv), (L, yl, xl), (R, yr, xr)):
            D[s, :a], D[s, a:], D[s + P, a:] = y[s, :a], x[s, a:], x[s, a:]
    return V, L, (R if want_right else None), starts


def drive(vp, fs, B, V, L, R, calls, items, resets=None, sched=None, workspace_bytes=0, reserve=None, mode=None, path="host"):
    """Process calls of calls[c] blocks, with engine-wide params sched[c] and eng.reset_streams(resets[c]) before call c.
    Returns per call {outL, outR, pf, vf} for every stream, and the number of passes."""
    S = V.shape[0]
    resets, sched = resets or {}, sched or {}
    eng = vp.Engine(fs, B, S, max(calls), workspace_bytes=workspace_bytes, reserve_orders=reserve)
    bufs = []
    try:
        if mode is not None:
            eng.set_mode(mode)
        eng.set_stream_params(0, items)
        if path == "device":
            n = V.shape[1]
            bufs = [eng.device_alloc(S * n * 4) for _ in range(5)]
            for p, a in zip(bufs, (V, L, R)):
                eng.h2d(p, np.ascontiguousarray(a))
        out, a = [], 0
        for c, nb in enumerate(calls):
            if c in sched:
                eng.set_params(vp.default_params(**sched[c]))
                eng.set_stream_params(0, items)
            if c in resets:
                eng.reset_streams(resets[c])
            x = slice(a * B, (a + nb) * B)
            if path == "host":
                l, r = eng.process(V[:, x], L[:, x], R[:, x] if R is not None else None)
            elif path == "pcm16":
                l, r = eng.process_pcm16(quant(V[:, x]), quant(L[:, x]), quant(R[:, x]) if R is not None else None)
            else:
                off = a * B * 4
                eng.process_device(nb, bufs[0] + off, bufs[1] + off, bufs[2] + off, bufs[3] + off, bufs[4] + off, V.shape[1])
                l = r = None
            out.append(dict(outL=None if l is None else l.copy(), outR=None if r is None else r.copy(),
                            pf=[[bytes(f) for f in eng.pitch_frames(s)] for s in range(S)],
                            frames=[eng.pitch_frames(s) for s in range(S)], vf=[eng.voc_frames(s) for s in range(S)]))
            a += nb
        if path == "device":
            oL, oR = np.zeros(V.shape, np.float32), np.zeros(V.shape, np.float32)
            eng.d2h(oL, bufs[3])
            eng.d2h(oR, bufs[4])
            a = 0
            for c, nb in enumerate(calls):
                out[c]["outL"], out[c]["outR"] = oL[:, a * B:(a + nb) * B], oR[:, a * B:(a + nb) * B]
                a += nb
        return out, -(-S // eng.info()["streams_per_pass"])
    finally:
        for p in bufs:
            eng.device_free(p)
        eng.close()


def same_stream(ca, sa, cb, sb):
    """stream sa of call record ca == stream sb of call record cb, bit for bit (audio and every frame record)"""
    if not (np.array_equal(ca["outL"][sa], cb["outL"][sb]) and np.array_equal(ca["outR"][sa], cb["outR"][sb])):
        return False
    if ca["pf"][sa] != cb["pf"][sb]:
        return False
    return all(np.array_equal(ca["vf"][sa][k], cb["vf"][sb][k]) for k in ("gated", "EeVoice", "EeSynth", "g"))


def assert_twins(out, P, reset_call, what):
    for s in range(P):
        for c in range(reset_call[s], len(out)):
            assert same_stream(out[c], s, out[c], s + P), "%s: stream %d != its twin %d in call %d" % (what, s, s + P, c)


def resets_from(reset_call):
    d = {}
    for s, c in enumerate(reset_call):
        d.setdefault(c, []).append(s)
    return d


def assert_audio(ref, got, what):
    sn, mx = snr_db(ref, got), maxabs(ref, got)
    assert sn >= SNR_MIN_DB and mx <= MAXABS_MAX, "%s: SNR %.1f dB, max abs err %.3e" % (what, sn, mx)


def ref_run(fs, B, v, l, r, params, schedule=None):
    """The reference's own C++ when it is built here, else the C oracle port (bit-identical to it)."""
    import oraclebind
    if refbind.available("strict"):
        return refbind.run(fs, B, v, l, synthR=r, params=params, log=True, schedule=schedule)
    return oraclebind.run(fs, B, v, l, synthR=r, params=params, log=True, schedule=schedule)


def assert_reference(vp, out, V, L, R, B, fs, starts, P, items, reset_call, sched_params=None, sched=None):
    """Each reset stream from its reset call on == the reference run on a zero prefix followed by the stream's X (which is
    the twin's input), audio within the stated tolerances and every pitch decision."""
    for s in range(P):
        c0 = reset_call[s]
        a = int(starts[c0])
        prm = dict(sched_params or {}, **items[s])
        schedule = None
        if sched:
            schedule = [(int(starts[c]) // B, refbind.default_params(**dict(q, **items[s]))) for c, q in sorted(sched.items()) if c > 0]
        r = ref_run(fs, B, V[s + P], L[s + P], None if R is None else R[s + P], refbind.default_params(**prm), schedule)
        gotL = np.concatenate([o["outL"][s] for o in out[c0:]])
        gotR = np.concatenate([o["outR"][s] for o in out[c0:]])
        what = "stream %d reset before call %d" % (s, c0)
        assert_audio(r["outL"][a:], gotL, what + " L")
        assert_audio(r["outR"][a:], gotR, what + " R")
        pre = sum(len(o["frames"][s + P]) for o in out[:c0])  # the twin's frames before the reset = the prefix's frames
        frames = [f for o in out[c0:] for f in o["frames"][s]]
        assert_decisions(compare_decisions(vp, oracle_decisions(r["pitch"])[pre:], frames), what)


def per_stream_bytes(vp, fs, B, S, calls):
    eng = vp.Engine(fs, B, S, max(calls))
    try:
        return eng.info()["workspace_bytes"] // S
    finally:
        eng.close()


# ---------------------------------------------------------------------------------------------------------- GPU tests
P13 = 13
TWIN_CONFIGS = {  # (fs, B, calls of different nBlocks, reset call of each of the 13 streams: three grid phases)
    "44k1_b1024": (44100.0, 1024, [19, 8, 14, 9, 25, 11]),
    "48k_b1024": (48000.0, 1024, [19, 8, 14, 9, 25, 11]),
    "48k_b128": (48000.0, 128, [150, 61, 97, 43, 180, 75]),
}
RESET_CALL = [1, 1, 1, 1, 2, 2, 2, 2, 4, 4, 4, 4, 4]


@pytest.fixture(scope="module", params=sorted(TWIN_CONFIGS))
def twin_run(request, vp):
    fs, B, calls = TWIN_CONFIGS[request.param]
    V, L, R, starts = twin_inputs(vp, fs, B, P13, calls, RESET_CALL)
    items = items_for(P13)
    per = per_stream_bytes(vp, fs, B, 2 * P13, calls)
    ws = 7 * per + per // 2  # passes of 7 streams: reset streams at both ends of a pass
    out, passes = drive(vp, fs, B, V, L, R, calls, items, resets=resets_from(RESET_CALL), workspace_bytes=ws, path="device")
    plain, _ = drive(vp, fs, B, V, L, R, calls, items, workspace_bytes=ws, path="device")
    return dict(name=request.param, fs=fs, B=B, calls=calls, V=V, L=L, R=R, starts=starts, items=items, out=out, plain=plain,
                passes=passes)


@pytest.mark.gpu
def test_reset_stream_equals_silent_twin_bitwise(twin_run):
    t = twin_run
    assert t["passes"] >= 3
    assert_twins(t["out"], P13, RESET_CALL, t["name"])
    # the old user was audible: without the reset the stream differs from its twin right after the handover
    for s in range(P13):
        assert not same_stream(t["plain"][RESET_CALL[s]], s, t["plain"][RESET_CALL[s]], s + P13), s


@pytest.mark.gpu
def test_streams_not_listed_are_untouched(twin_run):
    t = twin_run
    for c in range(len(t["calls"])):
        for s in range(P13, 2 * P13):
            assert same_stream(t["out"][c], s, t["plain"][c], s), "%s: stream %d call %d" % (t["name"], s, c)
        for s in range(P13):
            if c < RESET_CALL[s]:
                assert same_stream(t["out"][c], s, t["plain"][c], s), "%s: stream %d before its reset" % (t["name"], s)


@pytest.mark.gpu
def test_reset_stream_matches_reference_on_zero_prefix(vp, twin_run):
    t = twin_run
    assert_reference(vp, t["out"], t["V"], t["L"], t["R"], t["B"], t["fs"], t["starts"], P13, t["items"], RESET_CALL)


@pytest.mark.gpu
@pytest.mark.parametrize("B,calls,reset_call", [(1024, [10, 17, 15, 12, 20], 2), (128, [50, 70, 95, 66, 130], 2)])
def test_reset_at_aligned_block_is_a_fresh_instance(vp, B, calls, reset_call):
    """44.1 kHz: before block 27 (B = 1024, a multiple of 3) or 120 (B = 128, a multiple of 6) the grids are in their
    prepare phase, and the reset stream is a one-stream engine prepared fresh and fed only the new input."""
    fs, S = 44100.0, 3
    starts = np.concatenate([[0], np.cumsum(calls)]) * B
    a0 = int(starts[reset_call])
    assert a0 % (3 * 1024 if B == 1024 else 6 * 128) == 0
    n = int(starts[-1])
    V, L, R = vp.synth_host(fs, S, n, flavour=0, first_stream=4200)
    xv, xl, xr = vp.synth_host(fs, 1, n - a0, flavour=0, first_stream=4300)
    V[1, a0:], L[1, a0:], R[1, a0:] = xv[0], xl[0], xr[0]
    items = [dict(keyPitch=7), dict(DRY), dict(keyPitch=2, gainVoice=-20.0)]
    out, _ = drive(vp, fs, B, V, L, R, calls, items, resets={reset_call: [1]})
    eng = vp.Engine(fs, B, 1, max(calls), params=vp.default_params(**DRY))
    try:
        a = a0
        for c in range(reset_call, len(calls)):
            x = slice(a, a + calls[c] * B)
            l, r = eng.process(V[1:2, x], L[1:2, x], R[1:2, x])
            one = dict(outL=l, outR=r, pf=[[bytes(f) for f in eng.pitch_frames(0)]], vf=[eng.voc_frames(0)])
            assert same_stream(out[c], 1, one, 0), "call %d" % c
            a += calls[c] * B
    finally:
        eng.close()


@pytest.mark.gpu
def test_reset_around_bypass_and_order_changes(vp):
    """vocBool off for the block before the reset (the orphan store holds the old user's frames), pitchBool off around it
    (carried pitch frames with chunk limits) and an LPC order change: twin bit for bit, and the reference."""
    fs, B, P = 44100.0, 1024, 6
    calls = [17, 1, 2, 1, 9, 14, 12]
    base = dict(lpcVoice=40, lpcSynth=5)
    sched = {0: base, 1: dict(base, vocBool=0), 2: dict(base, pitchBool=0), 3: dict(base, pitchBool=0, lpcVoice=48, lpcSynth=8),
             4: dict(base, lpcVoice=48, lpcSynth=8), 5: dict(base, lpcVoice=32), 6: base}
    reset_call = [1, 2, 2, 3, 3, 4]
    V, L, R, starts = twin_inputs(vp, fs, B, P, calls, reset_call, first=4400)
    items = items_for(P)
    out, _ = drive(vp, fs, B, V, L, R, calls, items, resets=resets_from(reset_call), sched=sched, reserve=(48, 8))
    assert_twins(out, P, reset_call, "bypass / orders")
    assert_reference(vp, out, V, L, R, B, fs, starts, P, items, reset_call, sched_params=sched[0], sched=sched)


@pytest.mark.gpu
def test_reset_in_defined_mode(vp):
    fs, B, P = 44100.0, 1024, 5
    calls = [13, 7, 10, 22]
    reset_call = [1, 1, 2, 2, 3]
    V, L, R, _ = twin_inputs(vp, fs, B, P, calls, reset_call, first=4500)
    out, _ = drive(vp, fs, B, V, L, R, calls, items_for(P), resets=resets_from(reset_call), mode=vp.VP_MODE_DEFINED)
    assert_twins(out, P, reset_call, "defined mode")


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["host", "pcm16"])
def test_reset_on_host_paths(vp, path):
    """process_host / process_host_pcm16: the 26 streams move in slices of at most 9, so the reset streams 0..12 cross a
    slice boundary."""
    fs, B = 48000.0, 1024
    calls = [11, 6, 15, 9]
    reset_call = [1] * 5 + [2] * 4 + [3] * 4
    V, L, R, _ = twin_inputs(vp, fs, B, P13, calls, reset_call, first=4600)
    out, _ = drive(vp, fs, B, V, L, R, calls, items_for(P13), resets=resets_from(reset_call), path=path)
    assert_twins(out, P13, reset_call, path)


@pytest.mark.gpu
def test_reset_while_streaming(vp):
    """vp_engine_stream_block with resets between blocks at several block phases: twin bit for bit, and no graph capture
    beyond what the same run without resets makes."""
    fs, Bs, P, nb = 44100.0, 128, 4, 300
    reset_block = [37, 100, 161, 230]
    starts = np.arange(nb + 1) * Bs
    V, L, _, _ = twin_inputs(vp, fs, Bs, P, [1] * nb, reset_block, first=4700, want_right=False)
    items = [dict(it, gainSynth=-60.0) for it in items_for(P)]  # streaming carries side-chain channel 0 only

    def run(with_resets):
        eng = vp.Engine(fs, Bs, 2 * P, 1)
        try:
            eng.set_stream_params(0, items)
            hv, hs, ho = eng.stream_buffers()
            outs = []
            for b in range(nb):
                if with_resets:
                    eng.reset_streams([s for s in range(P) if reset_block[s] == b])
                hv[:] = V[:, starts[b]:starts[b + 1]]
                hs[:] = L[:, starts[b]:starts[b + 1]]
                eng.stream_block()
                outs.append(ho.copy())
            return np.concatenate(outs, axis=1), eng.stream_stats()["graph_captures"]
        finally:
            eng.close()
    out, cap = run(True)
    plain, cap0 = run(False)
    assert cap == cap0
    for s in range(P):
        a = reset_block[s] * Bs
        assert np.array_equal(out[s, a:], out[s + P, a:]), s
        assert np.array_equal(out[s, :a], plain[s, :a]), s
        assert np.array_equal(out[s + P], plain[s + P]), s


@pytest.mark.gpu
def test_reset_during_asynchronous_call(vp):
    """process_device without a sync, then reset_streams, then process_device: the first call is computed with the state
    it was issued with, the second shows the reset (== the stream had heard silence); duplicates and a repeated request act
    as one."""
    fs, B, S = 48000.0, 1024, 6
    n1, n2 = int(fs * 20.0) // B, 40
    n = (n1 + n2) * B
    voice, sl, _ = vp.synth_host(fs, S, n, flavour=0, first_stream=4800, want_right=False)
    silent = voice.copy(), sl.copy()
    for a in silent:
        a[[1, 4], :n1 * B] = 0.0

    def device_run(v, l, reset, sync_between):
        eng = vp.Engine(fs, B, S, n1)
        bufs = [eng.device_alloc(S * n * 4) for _ in range(3)]
        try:
            eng.h2d(bufs[0], v)
            eng.h2d(bufs[1], l)
            eng.process_device(n1, bufs[0], bufs[1], None, bufs[2], None, n, sync=sync_between)
            l0 = eng.stats()["kernel_launches"]
            for req in reset:
                eng.reset_streams(req)
            off = n1 * B * 4
            eng.process_device(n2, bufs[0] + off, bufs[1] + off, None, bufs[2] + off, None, n, sync=False)
            l1 = eng.stats()["kernel_launches"]
            eng.sync()
            out = np.zeros((S, n), np.float32)
            eng.d2h(out, bufs[2])
            return out, l1 - l0
        finally:
            for p in bufs:
                eng.device_free(p)
            eng.close()
    a, la = device_run(voice, sl, [[1, 4]], False)
    b, lb = device_run(voice, sl, [[1, 4]], True)
    c, lc = device_run(voice, sl, [[4, 1, 1], [4]], False)
    plain, lp = device_run(voice, sl, [], False)
    quiet, _ = device_run(silent[0], silent[1], [], False)
    assert np.array_equal(a, b) and np.array_equal(a, c)
    assert la == lb == lc == lp + 1
    assert np.array_equal(a[:, :n1 * B], plain[:, :n1 * B])
    for s in (1, 4):
        assert np.array_equal(a[s, n1 * B:], quiet[s, n1 * B:]), s
        assert not np.array_equal(a[s, n1 * B:], plain[s, n1 * B:]), s
    for s in (0, 2, 3, 5):
        assert np.array_equal(a[s], plain[s]), s


@pytest.mark.gpu
def test_reset_streams_cost_and_errors(vp):
    fs, B, S = 44100.0, 1024, 5
    nb = 8
    voice, sl, sr = vp.synth_host(fs, S, 4 * nb * B, flavour=0, first_stream=4900)
    items = items_for(3)[:S]
    x = [slice(k * nb * B, (k + 1) * nb * B) for k in range(4)]

    def run(actions):
        """four calls; actions[k](eng) before call k. Returns outputs and the kernel launches of each call."""
        eng = vp.Engine(fs, B, S, nb)
        try:
            eng.set_stream_params(0, items)
            outs, launches = [], []
            for k in range(4):
                if k in actions:
                    actions[k](eng)
                l0 = eng.stats()["kernel_launches"]
                outs.append(eng.process(voice[:, x[k]], sl[:, x[k]], sr[:, x[k]]))
                launches.append(eng.stats()["kernel_launches"] - l0)
            return outs, launches, eng.stream_params()
        finally:
            eng.close()
    plain, lp, _ = run({})
    # one reset: exactly one more launch in that call only; the key and gains are kept
    _, lr, params = run({2: lambda e: e.reset_streams([3])})
    assert lr == [lp[0], lp[1], lp[2] + 1, lp[3]]
    assert params == [vp.stream_params(**it).as_dict() for it in items]

    # an index out of range is VP_E_ARG and queues nothing (not even the valid entries before it)
    def bad(e):
        for req in ([0, S], [-1], [2, 0, 7]):
            with pytest.raises(vp.EngineError) as ei:
                e.reset_streams(req)
            assert ei.value.code == vp.VP_E_ARG
        arr = (C.c_int * 1)(0)
        assert e.lib.vp_engine_reset_streams(e.h, None, 1) == vp.VP_E_ARG
        assert e.lib.vp_engine_reset_streams(e.h, arr, -1) == vp.VP_E_ARG
        assert e.lib.vp_engine_reset_streams(e.h, None, 0) == vp.VP_OK
        e.reset_streams([])
    outs, lb, _ = run({1: bad})
    assert lb == lp
    for (l0, r0), (l1, r1) in zip(plain, outs):
        assert np.array_equal(l0, l1) and np.array_equal(r0, r1)

    # vp_engine_reset drops pending stream resets (no extra launch), and continues as after prepare
    def reset_all(e):
        e.reset_streams([0, 2])
        e.reset()
    outs, lz, _ = run({1: reset_all})
    fresh, lf, _ = run({1: lambda e: e.reset()})
    assert lz == lf
    for (l0, r0), (l1, r1) in zip(fresh, outs):
        assert np.array_equal(l0, l1) and np.array_equal(r0, r1)
    # before prepare
    lib = vp.load_library()
    h = C.c_void_p()
    assert lib.vp_engine_create(C.byref(h), 0) == vp.VP_OK
    try:
        assert lib.vp_engine_reset_streams(h, (C.c_int * 1)(0), 1) == vp.VP_E_STATE
    finally:
        lib.vp_engine_destroy(h)
