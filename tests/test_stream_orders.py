"""Per-stream vocoder LPC orders (vp_stream_orders, vp_engine_set_stream_orders, vp_engine_schedule_stream_orders): each stream
of a batch has its own lpcVoice / lpcSynth, set between calls or scheduled at any block.

CPU: the struct layouts match the header, the argument codes that need no device, and the read-site premise on the C
oracle: an order change scheduled at block b first changes the vocoder frame whose delayed start is the first in block b or
later. GPU: a batch with orders spread over <= 40 / <= 5 equals, bit for bit, each stream alone in an engine whose vp_params
carry its orders (also with >= 3 passes and with per-stream keys and gains); so does a batch above 40 on the generic
kernels; scheduled order changes give the same output in one call, cut at every event, cut at random and streamed block by
block; vocBool-off blocks (orphan frames), the host / device / PCM16 paths, reset_streams, set_params and the error codes
behave as documented; a uniform call launches what it launched before; streaming recaptures at most once. Against the
reference: every stream of the <= 40 / 5 batch, a mixed-tier batch, scheduled changes and the WAV manifest tokens."""
import ctypes as C
import json
import os
import shutil
import subprocess

import numpy as np
import pytest

import refbind
from common import assert_decisions, compare_decisions, oracle_decisions
from test_stream_schedule import assert_audio, assert_same, collect, device_call, finish, new_res, ref_run

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

LAYOUT_PROBE = r"""
#include <stddef.h>
#include <stdio.h>
#include "vp_engine.h"
int main(void) {
    printf("%zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(vp_stream_orders), offsetof(vp_stream_orders, lpcVoice),
           offsetof(vp_stream_orders, lpcSynth), sizeof(vp_stream_order_event), offsetof(vp_stream_order_event, stream),
           offsetof(vp_stream_order_event, reserved), offsetof(vp_stream_order_event, block), offsetof(vp_stream_order_event, o));
    return 0;
}
"""


# ---------------------------------------------------------------------------------------------------------- CPU
def test_layouts_match_header(vp, tmp_path):
    O, E = vp.StreamOrders, vp.StreamOrderEvent
    assert C.sizeof(O) == 8 and C.sizeof(E) == 24
    for name in ("vp_engine_set_stream_orders", "vp_engine_get_stream_orders", "vp_engine_schedule_stream_orders"):
        assert name in vp.ABI_SYMBOLS
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler to read the header's layout")
    src = tmp_path / "probe.c"
    src.write_text(LAYOUT_PROBE)
    exe = str(tmp_path / "probe")
    subprocess.check_call([cc, "-I", os.path.join(ROOT, "include"), "-o", exe, str(src)])
    got = [int(x) for x in subprocess.check_output([exe], text=True).split()]
    assert got == [C.sizeof(O), O.lpcVoice.offset, O.lpcSynth.offset, C.sizeof(E), E.stream.offset, E.reserved.offset,
                   E.block.offset, E.o.offset]


def test_null_engine_and_arguments(vp):
    lib = vp.load_library()
    o = (vp.StreamOrders * 1)(vp.StreamOrders(20, 3))
    ev = (vp.StreamOrderEvent * 1)()
    assert lib.vp_engine_set_stream_orders(None, 0, 1, o) == vp.VP_E_ARG
    assert lib.vp_engine_get_stream_orders(None, 0, 1, o) == vp.VP_E_ARG
    assert lib.vp_engine_schedule_stream_orders(None, ev, 1) == vp.VP_E_ARG
    assert lib.vp_engine_schedule_stream_orders(None, None, 0) == vp.VP_E_ARG


def _first_diff_frame(r0, r1):
    for k, (a, b) in enumerate(zip(r0["voc"], r1["voc"])):
        if (a.EeVoice, a.EeSynth, a.g) != (b.EeVoice, b.EeSynth, b.g):
            return k
    return None


@pytest.mark.parametrize("fs,B", [(44100.0, 1024), (48000.0, 1024), (44100.0, 128), (48000.0, 128)],
                         ids=["44k1-1024", "48k-1024", "44k1-128", "48k-128"])
def test_oracle_order_change_reaches_first_frame_of_block(vp, oracle, fs, B):
    """lpcVoice / lpcSynth changed at block b: the first vocoder frame record (EeVoice, EeSynth, g) that differs from a run
    without the change is the first frame whose delayed-timeline start lies in block b or later (frame k starts at k hopV
    while vocBool stays on)."""
    hop = oracle.sizes_for(fs, B)["hopV"]
    nb = 40 if B == 1024 else 300
    voice, sl, sr = vp.synth_host(fs, 1, nb * B, flavour=0, first_stream=5000)
    base = refbind.default_params()
    r0 = oracle.run(fs, B, voice[0], sl[0], synthR=sr[0], params=base, log=True)
    assert len(r0["voc"]) == -(-nb * B // hop)
    for b in (nb // 2, nb // 2 + 1, nb // 2 + 2):
        for new in (dict(lpcVoice=24), dict(lpcSynth=3), dict(lpcVoice=12, lpcSynth=2)):
            r1 = oracle.run(fs, B, voice[0], sl[0], synthR=sr[0], params=base, log=True,
                            schedule=[(b, refbind.default_params(**new))])
            assert _first_diff_frame(r0, r1) == -(-b * B // hop), (b, new)


# ---------------------------------------------------------------------------------------------------------- GPU helpers
def spread_orders(S, lo=(2, 2), hi=(40, 5)):
    """lpcVoice lo[0] .. hi[0] and lpcSynth lo[1] .. hi[1] spread over S streams (both ends included)."""
    v = np.linspace(lo[0], hi[0], S).round().astype(int)
    s = np.array([lo[1] + (k * 7) % (hi[1] - lo[1] + 1) for k in range(S)])
    s[0], s[-1] = lo[1], hi[1]
    return [(int(a), int(b)) for a, b in zip(v, s)]


def keys_gains(S, seed):
    rng = np.random.default_rng(seed)
    return [dict(keyPitch=int(rng.integers(0, 13)), gainVoc=float(rng.choice([-12.0, 0.0, 3.5])),
                 gainPitch=float(rng.choice([-6.0, 0.0, 3.0])), gainVoice=float(rng.choice([-60.0, -20.0])),
                 gainSynth=float(rng.choice([-60.0, -24.0]))) for _ in range(S)]


def batch_run(vp, fs, B, voice, sl, sr, orders, sp=None, workspace_bytes=0, reserve=None, path="host"):
    S, n = voice.shape
    eng = vp.Engine(fs, B, S, n // B, workspace_bytes=workspace_bytes, reserve_orders=reserve)
    res = new_res(S)
    try:
        if sp is not None:
            eng.set_stream_params(0, sp)
        eng.set_stream_orders(0, orders)
        if path == "host":
            l, r = eng.process(voice, sl, sr)
        else:
            l, r = device_call(eng, voice, sl, sr)
        collect(eng, S, res, l, r)
        res = finish(res)
        res["passes"] = -(-S // eng.info()["streams_per_pass"])
        res["orders"] = eng.stream_orders()
        return res
    finally:
        eng.close()


def solo_runs(vp, fs, B, voice, sl, sr, orders, sp=None):
    """Each stream alone in an engine whose vp_params carry its orders (and its key and gains)."""
    S, n = voice.shape
    res = new_res(S)
    outs = []
    for s in range(S):
        kw = dict(lpcVoice=orders[s][0], lpcSynth=orders[s][1])
        if sp is not None:
            kw.update(sp[s])
        eng = vp.Engine(fs, B, 1, n // B, params=vp.default_params(**kw))
        try:
            l, r = eng.process(voice[s:s + 1], sl[s:s + 1], sr[s:s + 1])
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


def reference_check(vp, fs, B, voice, sl, sr, res, params_of, schedule_of=None, streams=None):
    from concurrent.futures import ThreadPoolExecutor
    S = voice.shape[0]
    streams = list(range(S)) if streams is None else streams

    def one(s):
        return ref_run(fs, B, voice[s], sl[s], sr[s], params_of(s), schedule=schedule_of(s) if schedule_of else None)
    with ThreadPoolExecutor(max_workers=max(1, len(os.sched_getaffinity(0)))) as ex:
        refs = list(ex.map(one, streams))
    for s, r in zip(streams, refs):
        what = "stream %d" % s
        assert_audio(r["outL"], res["outL"][s], what + " L")
        assert_audio(r["outR"], res["outR"][s], what + " R")
        assert_decisions(compare_decisions(vp, oracle_decisions(r["pitch"]), res["frames"][s]), what)


# ---------------------------------------------------------------------------------------------------------- GPU: set between calls
@pytest.fixture(scope="module", params=[(44100.0, 1024, 45), (48000.0, 1024, 45)], ids=["44k1", "48k"])
def spread_case(request, vp):
    fs, B, nb = request.param
    S = 26
    voice, sl, sr = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=5100)
    orders = spread_orders(S)
    one = batch_run(vp, fs, B, voice, sl, sr, orders)
    return dict(fs=fs, B=B, nb=nb, S=S, voice=voice, sl=sl, sr=sr, orders=orders, one=one)


@pytest.mark.gpu
def test_batch_equals_each_stream_alone(vp, spread_case):
    c = spread_case
    args = (vp, c["fs"], c["B"], c["voice"], c["sl"], c["sr"], c["orders"])
    assert c["one"]["orders"] == [dict(lpcVoice=v, lpcSynth=s) for v, s in c["orders"]]
    assert_same(solo_runs(*args), c["one"], c["S"], "orders <= 40 / 5 against solo engines")


@pytest.mark.gpu
def test_batch_equals_alone_multi_pass_and_device(vp, spread_case):
    c = spread_case
    fs, B, S, nb = c["fs"], c["B"], c["S"], c["nb"]
    args = (vp, fs, B, c["voice"], c["sl"], c["sr"], c["orders"])
    eng = vp.Engine(fs, B, S, nb)
    per = eng.info()["workspace_bytes"] // S
    eng.close()
    multi = batch_run(*args, workspace_bytes=7 * per + per // 2)
    assert multi["passes"] >= 3
    assert_same(c["one"], multi, S, "%d passes" % multi["passes"])
    assert_same(c["one"], batch_run(*args, path="device"), S, "device path")


@pytest.mark.gpu
def test_batch_equals_alone_with_keys_and_gains(vp, spread_case):
    c = spread_case
    sp = keys_gains(c["S"], seed=int(c["fs"]))
    args = (vp, c["fs"], c["B"], c["voice"], c["sl"], c["sr"], c["orders"])
    assert_same(solo_runs(*args, sp=sp), batch_run(*args, sp=sp), c["S"], "orders, keys and gains per stream")


@pytest.mark.gpu
def test_spread_batch_matches_reference(vp, spread_case):
    c = spread_case
    reference_check(vp, c["fs"], c["B"], c["voice"], c["sl"], c["sr"], c["one"],
                    lambda s: refbind.default_params(lpcVoice=c["orders"][s][0], lpcSynth=c["orders"][s][1]))


@pytest.mark.gpu
def test_batch_above_40_equals_alone(vp):
    """All streams above 40 / 5 (within reserve_orders(64, 12)): the generic kernels, each frame at its own orders."""
    fs, B, nb, S = 48000.0, 1024, 30, 8
    voice, sl, sr = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=5200)
    orders = spread_orders(S, lo=(41, 6), hi=(64, 12))
    one = batch_run(vp, fs, B, voice, sl, sr, orders, reserve=(64, 12))
    assert_same(solo_runs(vp, fs, B, voice, sl, sr, orders), one, S, "orders > 40 against solo engines")


@pytest.mark.gpu
def test_mixed_tier_batch_matches_reference(vp):
    """Some streams above 40 / 5, the rest at or below, in one call: every stream matches the reference at its own orders."""
    fs, B, nb, S = 44100.0, 1024, 40, 10
    voice, sl, sr = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=5300)
    orders = spread_orders(S - 3) + [(64, 5), (48, 12), (40, 30)]
    one = batch_run(vp, fs, B, voice, sl, sr, orders, reserve=(64, 30))
    reference_check(vp, fs, B, voice, sl, sr, one, lambda s: refbind.default_params(lpcVoice=orders[s][0], lpcSynth=orders[s][1]))


# ---------------------------------------------------------------------------------------------------------- GPU: scheduled
def order_schedule(S, nb, seed, with_params=False):
    """Per stream: starting orders and 3-8 order events (<= 40 / 5) at its own blocks, including block 0 and the last block;
    with_params adds key / gain events at other blocks of the same streams."""
    rng = np.random.default_rng(seed)
    rnd = lambda: (int(rng.integers(2, 41)), int(rng.integers(2, 6)))
    base, events, pev = [rnd() for _ in range(S)], [], []
    for s in range(S):
        k = int(rng.integers(3, 9))
        blocks = {0, nb - 1}
        while len(blocks) < k:
            blocks.add(int(rng.integers(1, nb)))
        for b in sorted(blocks):
            events.append((s, b, rnd()))
        if with_params:
            for b in rng.choice(np.arange(1, nb), 3, replace=False):
                pev.append((s, int(b), dict(keyPitch=int(rng.integers(0, 13)), gainVoc=float(rng.choice([-9.0, 0.0])))))
    return base, events, pev


def orders_at(base, events, b):
    cur = list(base)
    for s, eb, o in sorted(events, key=lambda e: e[1]):
        if eb <= b:
            cur[s] = o
    return cur


def params_at(S, pev, b):
    cur = [vp_default_sp() for _ in range(S)]
    for s, eb, v in sorted(pev, key=lambda e: e[1]):
        if eb <= b:
            cur[s] = dict(cur[s], **v)
    return cur


def vp_default_sp():
    return dict(gainPitch=0.0, gainVoice=-60.0, gainSynth=-60.0, gainVoc=0.0, keyPitch=12)


def sched_run(vp, fs, B, voice, sl, sr, base, events, pev, cuts, mode):
    """mode "schedule": everything queued before the first call; "set": set_stream_orders / set_stream_params at every cut
    with the values in force there (the cuts must include every event block)."""
    S, n = voice.shape
    nb = n // B
    eng = vp.Engine(fs, B, S, nb)
    res = new_res(S)
    try:
        eng.set_stream_orders(0, base)
        if mode == "schedule":
            eng.schedule_stream_orders(events)
            if pev:
                eng.schedule_stream_params(pev)
        for a, b in zip(cuts, cuts[1:]):
            if mode == "set":
                eng.set_stream_orders(0, orders_at(base, events, a))
                if pev:
                    eng.set_stream_params(0, params_at(S, pev, a))
            x = slice(a * B, b * B)
            l, r = eng.process(voice[:, x], sl[:, x], sr[:, x])
            collect(eng, S, res, l, r)
        res = finish(res)
        res["orders"] = eng.stream_orders()
        return res
    finally:
        eng.close()


@pytest.fixture(scope="module", params=[(44100.0, 1024, 60, False), (48000.0, 128, 300, False), (48000.0, 1024, 60, True)],
                ids=["44k1-1024", "48k-128", "48k-1024-with-params"])
def sched_case(request, vp):
    fs, B, nb, with_params = request.param
    S = 26
    voice, sl, sr = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=5400)
    base, events, pev = order_schedule(S, nb, seed=int(fs) + B + with_params, with_params=with_params)
    one = sched_run(vp, fs, B, voice, sl, sr, base, events, pev, [0, nb], "schedule")
    return dict(fs=fs, B=B, nb=nb, S=S, voice=voice, sl=sl, sr=sr, base=base, events=events, pev=pev, one=one)


@pytest.mark.gpu
def test_scheduled_one_call_equals_any_cut(vp, sched_case):
    c = sched_case
    nb, S = c["nb"], c["S"]
    args = (vp, c["fs"], c["B"], c["voice"], c["sl"], c["sr"], c["base"], c["events"], c["pev"])
    ev_cuts = sorted({0, nb} | {b for _, b, _ in c["events"]} | {b for _, b, _ in c["pev"]})
    assert_same(c["one"], sched_run(*args, ev_cuts, "set"), S, "cut at every event with set_stream_orders")
    rng = np.random.default_rng(3)
    rnd = sorted({0, nb} | set(int(x) for x in rng.integers(1, nb, 6)))
    assert_same(c["one"], sched_run(*args, rnd, "schedule"), S, "cut at %r, schedule up front" % rnd)
    assert c["one"]["orders"] == [dict(lpcVoice=v, lpcSynth=s) for v, s in orders_at(c["base"], c["events"], nb - 1)]


@pytest.mark.gpu
def test_scheduled_streaming_block_by_block(vp, sched_case):
    """vp_engine_stream_block with the same schedule gives the one call's left output (the side-chain's right channel is not
    carried by streaming: the one call is run again without it)."""
    c = sched_case
    if c["pev"]:
        pytest.skip("parameter events are covered by test_stream_schedule")
    fs, B, nb, S = c["fs"], c["B"], c["nb"], c["S"]
    voice, sl = c["voice"], c["sl"]
    eng = vp.Engine(fs, B, S, nb)
    try:
        eng.set_stream_orders(0, c["base"])
        eng.schedule_stream_orders(c["events"])
        ref, _ = eng.process(voice, sl, None, want_right=False)
    finally:
        eng.close()
    eng = vp.Engine(fs, B, S, 1)
    out = np.zeros_like(voice)
    try:
        eng.set_stream_orders(0, c["base"])
        eng.schedule_stream_orders(c["events"])
        hv, hs, ho = eng.stream_buffers()
        for b in range(nb):
            hv[:] = voice[:, b * B:(b + 1) * B]
            hs[:] = sl[:, b * B:(b + 1) * B]
            eng.stream_block()
            out[:, b * B:(b + 1) * B] = ho
    finally:
        eng.close()
    assert np.array_equal(out, ref)


@pytest.mark.gpu
def test_scheduled_matches_reference(vp, sched_case):
    c = sched_case
    if c["B"] == 128:
        pytest.skip("one block size is enough against the reference; the cut tests cover B = 128 bit for bit")

    def start(s):
        first = [o for t, b, o in c["events"] if t == s and b == 0]
        return first[0] if first else c["base"][s]

    def params_of(s):
        o = start(s)
        return refbind.default_params(lpcVoice=o[0], lpcSynth=o[1])

    def schedule_of(s):
        blocks = sorted({b for t, b, _ in c["events"] if t == s and b > 0} | {b for t, b, _ in c["pev"] if t == s})
        out = []
        for b in blocks:
            o = orders_at([start(k) for k in range(c["S"])], [e for e in c["events"] if e[1] > 0], b)[s]
            kw = dict(params_at(c["S"], c["pev"], b)[s], lpcVoice=o[0], lpcSynth=o[1])
            out.append((b, refbind.default_params(**kw)))
        return out
    reference_check(vp, c["fs"], c["B"], c["voice"], c["sl"], c["sr"], c["one"], params_of, schedule_of)


# ---------------------------------------------------------------------------------------------------------- GPU: interplay
@pytest.mark.gpu
def test_voc_off_block_with_mixed_orders(vp):
    """A block with vocBool off between calls (its frames in flight finish from the orphan store) with per-stream orders that
    change across it: equals each stream alone with the same call sequence; host, PCM16 and device paths agree."""
    fs, B, S = 44100.0, 1024, 12
    calls = [(0, 7, 1), (7, 8, 0), (8, 9, 0), (9, 20, 1), (20, 21, 0), (21, 33, 1)]  # (first block, end, vocBool)
    nb = calls[-1][1]
    voice, sl, sr = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=5500)
    o1, o2 = spread_orders(S), spread_orders(S)[::-1]

    def run(S_, rows, orders_by_call, path="host"):
        eng = vp.Engine(fs, B, S_, nb)
        outL, outR = [], []
        try:
            for k, (a, b, voc) in enumerate(calls):
                eng.set_params(vp.default_params(vocBool=voc))
                eng.set_stream_orders(0, orders_by_call(k))
                x = slice(a * B, b * B)
                args = (voice[rows, x], sl[rows, x], sr[rows, x])
                if path == "pcm16":
                    q = lambda a_: np.clip(np.rint(a_ * np.float32(32768.0)), -32768, 32767).astype(np.int16)
                    l, r = eng.process_pcm16(*(q(a_) for a_ in args))
                elif path == "device":
                    l, r = device_call(eng, *(np.ascontiguousarray(a_) for a_ in args))
                else:
                    l, r = eng.process(*args)
                outL.append(l); outR.append(r)
        finally:
            eng.close()
        return np.concatenate(outL, axis=1), np.concatenate(outR, axis=1)
    by_call = lambda k: o1 if k < 3 else o2
    batch = run(S, slice(0, S), by_call)
    for s in range(S):
        solo = run(1, slice(s, s + 1), lambda k: [by_call(k)[s]])
        assert np.array_equal(solo[0][0], batch[0][s]) and np.array_equal(solo[1][0], batch[1][s]), "stream %d" % s
    dev = run(S, slice(0, S), by_call, path="device")
    assert np.array_equal(dev[0], batch[0]) and np.array_equal(dev[1], batch[1])
    p = run(S, slice(0, S), by_call, path="pcm16")
    for s in (0, S // 2, S - 1):
        solo = run(1, slice(s, s + 1), lambda k: [by_call(k)[s]], path="pcm16")
        assert np.array_equal(solo[0][0], p[0][s]), "pcm16 stream %d" % s


@pytest.mark.gpu
def test_reset_streams_and_set_params(vp):
    fs, B, S, nb = 44100.0, 1024, 5, 50
    voice, sl, sr = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=5600)
    base = spread_orders(S)
    ev = [(s, 25 + s, (12 + s, 3)) for s in range(S)] + [(s, 40, (30, 4)) for s in range(S)]

    def run(steps):
        eng = vp.Engine(fs, B, S, nb)
        L = []
        try:
            eng.set_stream_orders(0, base)
            for st in steps:
                if callable(st):
                    st(eng)
                else:
                    a, b = st
                    L.append(eng.process(voice[:, a * B:b * B], sl[:, a * B:b * B], sr[:, a * B:b * B])[0])
            return np.concatenate(L, axis=1), eng.stream_orders()
        finally:
            eng.close()
    sched = lambda evs: (lambda e: e.schedule_stream_orders(evs))
    # reset_streams keeps the listed stream's orders and drops its pending order events (the others keep theirs)
    a, oa = run([sched(ev), (0, 20), lambda e: e.reset_streams([1]), (20, nb)])
    b, ob = run([sched([x for x in ev if x[0] != 1]), (0, 20), lambda e: e.reset_streams([1]), (20, nb)])
    assert np.array_equal(a, b) and oa == ob
    assert oa[1] == dict(lpcVoice=base[1][0], lpcSynth=base[1][1])
    # set_params gives every stream its orders from the next block on; pending events still apply at their blocks
    P = vp.default_params(lpcVoice=22, lpcSynth=4)
    a, oa = run([sched(ev), (0, 20), lambda e: e.set_params(P), (20, nb)])
    steps = [(0, 20), lambda e: e.set_params(P)]
    cur = [(22, 4)] * S
    for lo, hi in zip([20, 25, 26, 27, 28, 29, 40], [25, 26, 27, 28, 29, 40, nb]):
        for s, blk, o in ev:
            if blk == lo:
                cur[s] = o
        steps += [(lambda v: (lambda e: e.set_stream_orders(0, v)))(list(cur)), (lo, hi)]
    b, ob = run(steps)
    assert np.array_equal(a, b) and oa == ob


@pytest.mark.gpu
def test_uniform_call_is_unchanged(vp):
    """A call in which every stream has the same orders launches what an engine that never set per-stream orders launches,
    with identical output: at the defaults and at 20 / 3 (set per stream vs. vp_params)."""
    fs, B, S, nb = 48000.0, 1024, 6, 30
    voice, sl, sr = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=5700)

    def run(params, orders):
        eng = vp.Engine(fs, B, S, nb, params=params)
        try:
            if orders is not None:
                eng.set_stream_orders(0, [orders] * S)
            k0 = eng.stats()["kernel_launches"]
            out = eng.process(voice, sl, sr)
            return eng.stats()["kernel_launches"] - k0, out
        finally:
            eng.close()
    k_plain, (l0, r0) = run(vp.default_params(), None)
    k_set, (l1, r1) = run(vp.default_params(), (40, 5))
    assert k_set == k_plain and np.array_equal(l0, l1) and np.array_equal(r0, r1)
    k_plain, (l0, r0) = run(vp.default_params(lpcVoice=20, lpcSynth=3), None)
    k_set, (l1, r1) = run(vp.default_params(), (20, 3))
    assert k_set == k_plain and np.array_equal(l0, l1) and np.array_equal(r0, r1)


@pytest.mark.gpu
def test_streaming_order_changes_cost_at_most_one_capture(vp):
    fs, B, S, nb = 44100.0, 128, 8, 150
    voice, sl, _ = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=5800, want_right=False)
    rng = np.random.default_rng(17)

    def run(changes):
        eng = vp.Engine(fs, B, S, 1)
        try:
            hv, hs, _ = eng.stream_buffers()
            for b in range(nb):
                if b in changes:
                    eng.set_stream_orders(0, changes[b])
                hv[:] = voice[:, b * B:(b + 1) * B]
                hs[:] = sl[:, b * B:(b + 1) * B]
                eng.stream_block()
            return eng.stream_stats()["graph_captures"]
        finally:
            eng.close()
    plain = run({})
    mixed = lambda: [(int(rng.integers(2, 41)), int(rng.integers(2, 6))) for _ in range(S)]
    once = run({10: mixed()})
    many = run({b: mixed() for b in (10, 40, 41, 77, 120)})
    # the switch to mixed orders captures each block phase once more; later changes among orders <= 40 / 5 capture nothing
    assert plain < once <= 2 * plain and many == once


@pytest.mark.gpu
def test_errors_change_nothing(vp):
    fs, B, S = 44100.0, 1024, 4
    lib = vp.load_library()
    h = C.c_void_p()
    assert lib.vp_engine_create(C.byref(h), 0) == vp.VP_OK
    try:
        o = (vp.StreamOrders * 1)(vp.StreamOrders(20, 3))
        assert lib.vp_engine_set_stream_orders(h, 0, 1, o) == vp.VP_E_STATE
        assert lib.vp_engine_get_stream_orders(h, 0, 1, o) == vp.VP_E_STATE
        assert lib.vp_engine_schedule_stream_orders(h, (vp.StreamOrderEvent * 1)(), 1) == vp.VP_E_STATE
    finally:
        lib.vp_engine_destroy(h)
    eng = vp.Engine(fs, B, S, 10)
    try:
        before = eng.stream_orders()
        for first, items, code in [(0, [(20, 3), (101, 3)], vp.VP_E_RANGE), (0, [(20, 3), (20, 31)], vp.VP_E_RANGE),
                                   (0, [(1, 3)], vp.VP_E_RANGE), (0, [(20, 3), (41, 5)], vp.VP_E_STATE),
                                   (0, [(20, 6)], vp.VP_E_STATE), (S - 1, [(20, 3), (20, 3)], vp.VP_E_ARG),
                                   (-1, [(20, 3)], vp.VP_E_ARG)]:
            with pytest.raises(vp.EngineError) as ei:
                eng.set_stream_orders(first, items)
            assert ei.value.code == code, (first, items)
            assert eng.stream_orders() == before
        assert lib.vp_engine_set_stream_orders(eng.h, 0, 1, None) == vp.VP_E_ARG
        good = (0, 5, (20, 3))
        for bad, code in [([good, (1, 6, (2, 31))], vp.VP_E_RANGE), ([good, (1, 6, (64, 5))], vp.VP_E_STATE),
                          ([good, (S, 6, (20, 3))], vp.VP_E_ARG), ([good, (0, -1, (20, 3))], vp.VP_E_ARG)]:
            with pytest.raises(vp.EngineError) as ei:
                eng.schedule_stream_orders(bad)
            assert ei.value.code == code
        assert lib.vp_engine_schedule_stream_orders(eng.h, None, 1) == vp.VP_E_ARG
        assert lib.vp_engine_schedule_stream_orders(eng.h, (vp.StreamOrderEvent * 1)(), -1) == vp.VP_E_ARG
        voice, sl, sr = vp.synth_host(fs, S, 10 * B, flavour=0, first_stream=5900)
        l1, _ = eng.process(voice, sl, sr)
        assert eng.stream_orders() == before
    finally:
        eng.close()
    eng = vp.Engine(fs, B, S, 10)
    try:
        l0, _ = eng.process(voice, sl, sr)
    finally:
        eng.close()
    assert np.array_equal(l0, l1)


@pytest.mark.gpu
def test_wav_manifest_order_tokens(vp, tmp_path):
    """lpcVoice= / lpcSynth= on manifest lines: each job runs at its own orders (one above 40, reserved from the manifest) and
    matches the reference at those orders."""
    from test_wav import read_f32, write_f32
    from vocoderproject_b200 import build as b
    b.build()
    tool = b.build_wavbatch()
    fs, B, K, n = 44100.0, 1024, 8, 60000
    v, l, r = vp.synth_host(fs, 3, n, flavour=0, first_stream=6000)
    toks = ["lpcVoice=12 lpcSynth=2", "", "lpcVoice=56 lpcSynth=9 key=3"]
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
    params = [dict(lpcVoice=12, lpcSynth=2), dict(), dict(lpcVoice=56, lpcSynth=9, keyPitch=3)]
    for s in range(3):
        _, x = read_f32(str(tmp_path / ("o%d.wav" % s)))
        ref = ref_run(fs, B, v[s], l[s], r[s], refbind.default_params(**params[s]))
        m = len(x) // B * B
        assert_audio(ref["outL"][:m], x[:m, 0], "job %d L" % s)
        assert_audio(ref["outR"][:m], x[:m, 1], "job %d R" % s)
