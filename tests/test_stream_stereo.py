"""Stereo streaming (vp_engine_stream_buffers_stereo): vp_engine_stream_block with the right side-chain and the right output.

From the first call of the stereo getter on, every block equals vp_engine_process_host(e, 1, voice, synthL, synthR, outL,
outR, B) bit for bit, whatever each stream's dry side-chain does; blocks streamed in mono before keep their meaning (right
channel = left channel). An engine that never asks for stereo streams as before and refuses the dry side-chain.
CPU: the entry point refuses a null engine.
GPU: block-by-block identity with the host path at two rates and block sizes over several passes, automation of the dry
side-chain (set and scheduled) without new graph captures once every block phase has been seen, the right history across
the mono -> stereo switch (host path and C oracle), the mono path, per-stream resets and snapshots, and prepare."""
import ctypes as C

import numpy as np
import pytest

import refbind
from common import MAXABS_MAX, SNR_MIN_DB, assert_decisions, compare_decisions, maxabs, oracle_decisions, snr_db
from test_stream_params import spread


# ---------------------------------------------------------------------------------------------------------- CPU
def test_stereo_buffers_null_engine_is_arg(vp):
    lib = vp.load_library()
    p = [C.c_void_p() for _ in range(5)]
    assert lib.vp_engine_stream_buffers_stereo(None, *[C.byref(x) for x in p]) == vp.VP_E_ARG
    assert lib.vp_engine_stream_buffers_stereo(None, None, None, None, None, None) == vp.VP_E_ARG
    assert "vp_engine_stream_buffers_stereo" in vp.ABI_SYMBOLS


# ---------------------------------------------------------------------------------------------------------- GPU helpers
def several_pass_workspace(vp, fs, B, S, passes=4):
    """A workspace that makes the engine run S streams in about `passes` passes."""
    eng = vp.Engine(fs, B, S, 1)
    per = eng.info()["workspace_bytes"] // S
    eng.close()
    return (S // passes) * per + per // 2


class Twins:
    """A stereo streaming engine and a host-path engine (one process call per block) given the same inputs and changes."""

    def __init__(self, vp, fs, B, S, items=None, workspace_bytes=0, host_blocks=1):
        self.B = B
        self.eng = vp.Engine(fs, B, S, 1, workspace_bytes=workspace_bytes)
        self.ref = vp.Engine(fs, B, S, host_blocks, workspace_bytes=workspace_bytes)
        if items is not None:
            self.both("set_stream_params", 0, items)
        self.hv, self.hs, self.hr, self.ho, self.hor = self.eng.stream_buffers(stereo=True)

    def both(self, name, *args):
        getattr(self.eng, name)(*args)
        getattr(self.ref, name)(*args)

    def block(self, V, L, R, b):
        """Block b through both engines: (stream outL, stream outR, host outL, host outR)."""
        x = slice(b * self.B, (b + 1) * self.B)
        rl, rr = self.ref.process(V[:, x], L[:, x], R[:, x])
        self.hv[:], self.hs[:], self.hr[:] = V[:, x], L[:, x], R[:, x]
        self.eng.stream_block()
        return self.ho.copy(), self.hor.copy(), rl, rr

    def close(self):
        self.eng.close()
        self.ref.close()


# ---------------------------------------------------------------------------------------------------------- GPU tests
@pytest.mark.gpu
@pytest.mark.parametrize("fs,B,nb", [(44100.0, 128, 150), (48000.0, 1024, 40)], ids=["44k1_b128", "48k_b1024"])
def test_stereo_stream_equals_host_path_block_by_block(vp, fs, B, nb):
    """Per-stream keys and gains including gainSynth at -59.0 (off) / -58.9 (on), dry voice on some streams, several passes:
    outL and outR of every block equal process(voice, synthL, synthR) one block per call, and L == R exactly for every
    stream whose dry side-chain is off."""
    S = 26
    V, L, R = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=7000)
    items = spread(S)
    assert any(it["gainSynth"] == -58.9 for it in items) and any(it["gainSynth"] == -59.0 for it in items)
    t = Twins(vp, fs, B, S, items, workspace_bytes=several_pass_workspace(vp, fs, B, S))
    try:
        assert -(-S // t.eng.info()["streams_per_pass"]) >= 3
        outL, outR = [], []
        for b in range(nb):
            sl, sr, rl, rr = t.block(V, L, R, b)
            assert np.array_equal(sl, rl), "block %d outL" % b
            assert np.array_equal(sr, rr), "block %d outR" % b
            outL.append(sl)
            outR.append(sr)
        assert t.eng.stream_stats()["graph_launches"] == nb
    finally:
        t.close()
    outL, outR = np.concatenate(outL, axis=1), np.concatenate(outR, axis=1)
    for s, it in enumerate(items):
        assert np.array_equal(outL[s], outR[s]) == (it["gainSynth"] <= -59.0), s
        assert np.any(outL[s] != 0.0) == (s != S - 1), s  # (the last stream has every path at -60 / -59.5 dB: off)


@pytest.mark.gpu
def test_stereo_dry_sidechain_automation_without_new_captures(vp):
    """gainSynth switched on and off for some streams mid-run, through set_stream_params and schedule_stream_params, both
    engines given the same changes: equal block by block. Blocks 0..79 see every block phase with no stream's dry
    side-chain on and with one on; after that no block adds a graph capture, whatever the gains do."""
    fs, B, S, nb = 44100.0, 128, 8, 200
    V, L, R = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=7100)
    start = [dict(keyPitch=(3 * s) % 13, gainVoc=-2.0 * s, gainPitch=1.0 - s) for s in range(S)]
    on, off = dict(gainSynth=-10.0), dict(gainSynth=-60.0)
    sets = {40: {2: on}, 135: {5: dict(gainSynth=-3.0), 1: dict(gainSynth=-58.9)}, 170: {0: on}, 185: {3: dict(gainVoc=4.0)}}
    scheds = {60: [(2, 80, off)], 110: [(5, 120, dict(gainSynth=-20.0))], 140: [(5, 150, off), (1, 150, dict(gainSynth=-59.0))],
              145: [(6, 160, dict(keyPitch=1, gainVoc=-9.0))]}
    t = Twins(vp, fs, B, S, start)
    flags = []
    try:
        captures = None
        for b in range(nb):
            for s, d in sets.get(b, {}).items():
                t.both("set_stream_params", s, [d])
            if b in scheds:
                t.both("schedule_stream_params", scheds[b])
            if b == 80:
                captures = t.eng.stream_stats()["graph_captures"]
            sl, sr, rl, rr = t.block(V, L, R, b)
            assert np.array_equal(sl, rl) and np.array_equal(sr, rr), "block %d" % b
            flags.append(any(p["gainSynth"] > -59.0 for p in t.eng.stream_params()))
        st = t.eng.stream_stats()
        assert st["graph_launches"] == nb and st["graph_captures"] == captures
    finally:
        t.close()
    # the flag really was off and on in both stretches, and flipped after block 80 as planned
    assert not any(flags[:40]) and all(flags[40:80]) and not any(flags[80:120]) and all(flags[120:150])
    assert not any(flags[150:170]) and all(flags[170:])


@pytest.mark.gpu
def test_right_history_across_the_switch(vp, oracle):
    """k blocks with the mono buffers (dry side-chain off), then stereo, then gainSynth on for one stream a few blocks
    later, while the delayed timeline still reads mono-era input: equal to the host path fed synthR = synthL for the
    first k blocks and synthR afterwards (and not to one fed synthR throughout); for three streams the whole run also
    matches the C oracle on that right channel with that gainSynth schedule."""
    fs, B, S, nb, k, t_on = 44100.0, 128, 4, 420, 30, 36
    V, L, R = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=7200)
    Rcat = R.copy()
    Rcat[:, :k * B] = L[:, :k * B]
    items = [dict(keyPitch=s * 3, gainVoc=-3.0 * s, gainVoice=-20.0 if s == 3 else -60.0) for s in range(S)]
    on_stream, on = 1, dict(gainSynth=-6.0)
    eng = vp.Engine(fs, B, S, 1)
    outL, outR, frames = [], [], [[] for _ in range(S)]
    try:
        eng.set_stream_params(0, items)
        hv, hs, ho = eng.stream_buffers()
        hr = hor = None
        for b in range(nb):
            if b == k:
                hv2, hs2, hr, ho2, hor = eng.stream_buffers(stereo=True)
                assert hv2.ctypes.data == hv.ctypes.data and hs2.ctypes.data == hs.ctypes.data and ho2.ctypes.data == ho.ctypes.data
            if b == t_on:
                eng.set_stream_params(on_stream, [on])
            x = slice(b * B, (b + 1) * B)
            hv[:], hs[:] = V[:, x], L[:, x]
            if hr is not None:
                hr[:] = R[:, x]
            eng.stream_block()
            outL.append(ho.copy())
            outR.append(hor.copy() if hor is not None else ho.copy())
            for s in range(S):
                frames[s] += eng.pitch_frames(s)
    finally:
        eng.close()
    outL, outR = np.concatenate(outL, axis=1), np.concatenate(outR, axis=1)

    def host(right):
        h = vp.Engine(fs, B, S, nb)
        try:
            h.set_stream_params(0, items)
            l1, r1 = h.process(V[:, :t_on * B], L[:, :t_on * B], right[:, :t_on * B])
            h.set_stream_params(on_stream, [on])
            l2, r2 = h.process(V[:, t_on * B:], L[:, t_on * B:], right[:, t_on * B:])
            return np.concatenate([l1, l2], axis=1), np.concatenate([r1, r2], axis=1)
        finally:
            h.close()
    hl, hr_ = host(Rcat)
    assert np.array_equal(outL, hl) and np.array_equal(outR, hr_)
    _, wrong = host(R)
    assert not np.array_equal(outR[on_stream], wrong[on_stream])  # the mono-era right history is heard
    for s in range(S):
        assert np.array_equal(outL[s], outR[s]) == (s != on_stream), s
    for s in (0, on_stream, 3):
        prm = refbind.default_params(**items[s])
        sched = [(t_on, refbind.default_params(**dict(items[s], **on)))] if s == on_stream else None
        r = oracle.run(fs, B, V[s], L[s], synthR=Rcat[s], params=prm, log=True, schedule=sched)
        for ch, got in (("outL", outL[s]), ("outR", outR[s])):
            sn, mx = snr_db(r[ch], got), maxabs(r[ch], got)
            assert sn >= SNR_MIN_DB and mx <= MAXABS_MAX, "stream %d %s: SNR %.1f dB, max abs err %.3e" % (s, ch, sn, mx)
        assert_decisions(compare_decisions(vp, oracle_decisions(r["pitch"]), frames[s]), "stream %d" % s)


@pytest.mark.gpu
def test_mono_streaming_is_untouched(vp):
    """An engine that never asks for stereo still refuses a dry side-chain (also one scheduled for a later block). Either
    getter may come first: both return the same three mono buffers; the right buffers start at zero."""
    fs, B, S = 44100.0, 128, 3
    eng = vp.Engine(fs, B, S, 1)
    try:
        hv, hs, ho = eng.stream_buffers()
        eng.stream_block()
        eng.schedule_stream_params([(1, 2, dict(gainSynth=-10.0))])
        eng.stream_block()
        with pytest.raises(vp.EngineError) as ei:
            eng.stream_block()
        assert ei.value.code == vp.VP_E_ARG
        sv, ss, sr, so, sor = eng.stream_buffers(stereo=True)
        assert [a.ctypes.data for a in (sv, ss, so)] == [a.ctypes.data for a in (hv, hs, ho)]
        assert not np.any(sr) and not np.any(sor)
        mv, ms, mo = eng.stream_buffers()
        assert [a.ctypes.data for a in (mv, ms, mo)] == [a.ctypes.data for a in (hv, hs, ho)]
        eng.stream_block()  # stereo now: the dry side-chain is streamed
    finally:
        eng.close()
    eng = vp.Engine(fs, B, S, 1)
    try:
        sv, ss, sr, so, sor = eng.stream_buffers(stereo=True)
        mv, ms, mo = eng.stream_buffers()
        assert [a.ctypes.data for a in (mv, ms, mo)] == [a.ctypes.data for a in (sv, ss, so)]
        assert len({a.ctypes.data for a in (sv, ss, sr, so, sor)}) == 5
        sv2, ss2, sr2, so2, sor2 = eng.stream_buffers(stereo=True)
        assert [a.ctypes.data for a in (sv2, ss2, sr2, so2, sor2)] == [a.ctypes.data for a in (sv, ss, sr, so, sor)]
    finally:
        eng.close()


@pytest.mark.gpu
def test_stereo_resets_and_snapshots(vp):
    """reset_streams between stereo blocks equals the host path with the same resets; a stream saved from the stereo
    streaming engine and loaded into a fresh engine continues, on process(voice, synthL, synthR), bit for bit as in its
    uninterrupted run."""
    fs, B, S, nb, t_save = 44100.0, 128, 6, 160, 70
    V, L, R = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=7300)
    items = [dict(keyPitch=s * 2, gainVoc=-1.0 * s, gainSynth=-12.0 if s % 2 else -60.0, gainVoice=-25.0 if s == 4 else -60.0)
             for s in range(S)]
    resets = {45: [1, 2], 101: [3], 121: [1, 4, 5]}
    t = Twins(vp, fs, B, S, items)
    outL, outR = [], []
    try:
        for b in range(nb):
            if b in resets:
                t.both("reset_streams", resets[b])
            if b == t_save:
                blob = t.eng.save_streams([3])
            sl, sr, rl, rr = t.block(V, L, R, b)
            assert np.array_equal(sl, rl) and np.array_equal(sr, rr), "block %d" % b
            outL.append(sl)
            outR.append(sr)
    finally:
        t.close()
    outL, outR = np.concatenate(outL, axis=1), np.concatenate(outR, axis=1)
    # stream 3 from t_save up to its reset at block 101
    end = 101
    fresh = vp.Engine(fs, B, 1, end - t_save)
    try:
        fresh.load_streams([0], blob)
        x = slice(t_save * B, end * B)
        l, r = fresh.process(V[3:4, x], L[3:4, x], R[3:4, x])
    finally:
        fresh.close()
    assert np.array_equal(l[0], outL[3, x]) and np.array_equal(r[0], outR[3, x])
    assert not np.array_equal(l[0], r[0])  # stream 3 has the dry side-chain on: its right channel is its own


@pytest.mark.gpu
def test_prepare_ends_stereo(vp):
    """vp_engine_prepare frees every streaming buffer: stream_block is VP_E_STATE until a getter is called again, and after
    the mono getter the engine streams in mono (the dry side-chain is refused again). Before prepare the stereo getter is
    VP_E_STATE."""
    fs, B, S = 44100.0, 128, 2
    lib = vp.load_library()
    h = C.c_void_p()
    assert lib.vp_engine_create(C.byref(h), 0) == vp.VP_OK
    try:
        p = [C.c_void_p() for _ in range(5)]
        assert lib.vp_engine_stream_buffers_stereo(h, *[C.byref(x) for x in p]) == vp.VP_E_STATE
    finally:
        lib.vp_engine_destroy(h)
    eng = vp.Engine(fs, B, S, 1)
    try:
        eng.set_stream_params(0, [dict(gainSynth=-10.0)] * S)
        eng.stream_buffers(stereo=True)
        eng.stream_block()
        assert lib.vp_engine_prepare(eng.h, fs, B, S, 1, 0) == vp.VP_OK
        with pytest.raises(vp.EngineError) as ei:
            eng.stream_block()
        assert ei.value.code == vp.VP_E_STATE
        eng.set_stream_params(0, [dict(gainSynth=-10.0)] * S)
        eng.stream_buffers()
        with pytest.raises(vp.EngineError) as ei:
            eng.stream_block()
        assert ei.value.code == vp.VP_E_ARG
        eng.stream_buffers(stereo=True)
        eng.stream_block()
    finally:
        eng.close()
