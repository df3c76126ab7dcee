"""Per-stream state snapshots (vp_engine_snapshot_size / _save_streams / _load_streams).

A saved stream loaded into another slot -- of the same engine, of an engine at the same grid phase, or of a freshly
prepared engine of another size -- continues bit for bit as the stream would have without interruption (its "twin"):
audio, every pitch record and every vocoder frame record. The source is untouched, a blob that fails any check is refused
before anything reaches the GPU, and the engine then continues as if it had never seen the call.
CPU: the ABI names, the null-engine codes and the documented layout.
GPU: moves within an engine (several rates, block sizes, bypass stretches, per-stream values, modes and process paths),
between engines, checkpoint / resize, the reference anchor, ordering against asynchronous calls, resets, events and
streaming graphs, and rejection without side effects."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import refbind
from common import MAXABS_MAX, SNR_MIN_DB, assert_decisions, compare_decisions, maxabs, oracle_decisions, snr_db

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------------------------------------------------- layout
def units_per_stream(sizes, block, history, cap_v, cap_s):
    """16-byte units of one stream's raw state, segment by segment as the header documents them."""
    gate_carry = sizes["inSize"] // block + 1
    segs = [("hist", 3 * history * 4), ("gate", gate_carry * 4 * 8), ("cAV", 4 * (cap_v + 1) * 8), ("cAS", 4 * (cap_s + 1) * 8),
            ("cEeS", 4 * 8), ("cG", 4 * 8), ("gainHist", 20 * 8), ("frames", 2 * 240), ("marks", 304), ("chunkGains", 2 * 4 * 4),
            ("oAV", 8 * (cap_v + 1) * 8), ("oAS", 8 * (cap_s + 1) * 8), ("oEeS", 8 * 8), ("oG", 8 * 8)]
    off, table = 0, {}
    for name, b in segs:
        assert b % 16 == 0
        table[name] = off
        off += b
    return off // 16, table


def fnv64(data):
    """FNV-1a 64 over little-endian 64-bit words (the snapshot checksums)."""
    h, m = 14695981039346656037, (1 << 64) - 1
    for w in np.frombuffer(data, dtype="<u8").tolist():
        h = ((h ^ w) * 1099511628211) & m
    return h


def fix_record_checksum(blob, k, rec_bytes, vp):
    b = bytearray(blob)
    r0 = vp.VP_SNAPSHOT_HEADER_BYTES + k * rec_bytes
    b[r0:r0 + 8] = bytes(8)
    b[r0:r0 + 8] = fnv64(bytes(b[r0:r0 + rec_bytes])).to_bytes(8, "little")
    return bytes(b)


# ---------------------------------------------------------------------------------------------------------- CPU
def test_snapshot_abi_names_resolve(vp):
    lib = vp.load_library()
    for name in ("vp_engine_snapshot_size", "vp_engine_save_streams", "vp_engine_load_streams"):
        assert hasattr(lib, name) and name in vp.ABI_SYMBOLS


def test_snapshot_null_engine_codes(vp):
    lib = vp.load_library()
    arr = (C.c_int * 1)(0)
    n = C.c_size_t(0)
    buf = C.create_string_buffer(4096)
    assert lib.vp_engine_snapshot_size(None, 1, C.byref(n)) == vp.VP_E_ARG
    assert lib.vp_engine_save_streams(None, arr, 1, buf, 4096) == vp.VP_E_ARG
    assert lib.vp_engine_load_streams(None, arr, 1, buf.raw, 4096) == vp.VP_E_ARG


def test_snapshot_layout_constants_match_header(vp):
    src = open(os.path.join(ROOT, "include", "vp_engine.h")).read()
    got = {k: int(v) for k, v in re.findall(r"#define (VP_SNAPSHOT_\w+) (\d+)", src)}
    assert got == {"VP_SNAPSHOT_VERSION": vp.VP_SNAPSHOT_VERSION, "VP_SNAPSHOT_HEADER_BYTES": vp.VP_SNAPSHOT_HEADER_BYTES,
                   "VP_SNAPSHOT_RECORD_BYTES": vp.VP_SNAPSHOT_RECORD_BYTES}
    # fixed record part: checksum, vp_stream_params, vp_stream_orders, lpcPitch in force / next, 24 row orders, reserved
    assert vp.VP_SNAPSHOT_RECORD_BYTES == 8 + C.sizeof(vp.StreamParams) + C.sizeof(vp.StreamOrders) + 8 + 24 * 4 + 4
    # about 43 KB of raw state per stream at 48 kHz (rows for orders 40 / 5)
    z = vp.sizes_for(48000.0, 1024)
    history = (z["latency"] + z["frameLenP"] + 3 * z["chunk"] + 100 + 3) & ~3
    units, _ = units_per_stream(z, 1024, history, 40, 5)
    assert 40000 < units * 16 < 46000


def test_snapshot_checksum_detects_any_single_byte(vp):
    rng = np.random.default_rng(1)
    data = rng.integers(0, 256, 4096, dtype=np.uint8).tobytes()
    h = fnv64(data)
    for pos in (0, 7, 8, 2047, 4095):
        b = bytearray(data)
        b[pos] ^= 0x10
        assert fnv64(bytes(b)) != h


# ---------------------------------------------------------------------------------------------------------- GPU helpers
def quant(a):
    return np.clip(np.rint(a * np.float32(32768.0)), -32768, 32767).astype(np.int16)


ITEMS = [dict(keyPitch=4, gainVoc=-3.0, gainPitch=1.0, gainVoice=-14.0, gainSynth=-60.0),
         dict(keyPitch=9, gainVoc=0.0, gainPitch=-2.0, gainVoice=-60.0, gainSynth=-18.0),
         dict(keyPitch=12, gainVoc=-6.0, gainPitch=0.0, gainVoice=-60.0, gainSynth=-60.0),
         dict(keyPitch=1, gainVoc=-1.5, gainPitch=3.0, gainVoice=-20.0, gainSynth=-25.0)]
ORDERS = [(40, 5), (20, 5), (64, 8), (32, 3)]
PITCH = [15, 8, 24, 15]
RESERVE, RESERVE_P = (64, 8), 24


class Run:
    """One engine with per-slot values mirrored on the host (set_params broadcasts; the mirror puts them back)."""

    def __init__(self, vp, fs, B, S, max_blocks, items, orders, pitch, mode=None, workspace_bytes=0):
        self.vp, self.B, self.S = vp, B, S
        self.eng = vp.Engine(fs, B, S, max_blocks, workspace_bytes=workspace_bytes, reserve_orders=RESERVE,
                             reserve_pitch_order=RESERVE_P)
        if mode is not None:
            self.eng.set_mode(mode)
        self.items, self.orders = [dict(it) for it in items], [tuple(o) for o in orders]
        self.eng.set_stream_pitch_orders(0, pitch)
        self.push()
        self.b0 = 0

    def push(self):
        self.eng.set_stream_params(0, self.items)
        self.eng.set_stream_orders(0, self.orders)

    def toggles(self, **q):
        self.eng.set_params(self.vp.default_params(**q))
        self.push()

    def took(self, slots, src_items, src_orders):
        """after a load: the mirror of the loaded slots, and a check that the engine gave them the record's values"""
        for s, it, o in zip(slots, src_items, src_orders):
            self.items[s], self.orders[s] = dict(it), tuple(o)
            assert self.eng.stream_params(s, 1)[0] == self.vp.stream_params(**it).as_dict()
            assert self.eng.stream_orders(s, 1)[0] == {"lpcVoice": o[0], "lpcSynth": o[1]}

    def call(self, V, L, R, nb, path="host"):
        eng, B, S = self.eng, self.B, self.S
        x = slice(self.b0 * B, (self.b0 + nb) * B)
        v, l = np.ascontiguousarray(V[:, x]), np.ascontiguousarray(L[:, x])
        r = None if R is None else np.ascontiguousarray(R[:, x])
        if path == "host":
            oL, oR = eng.process(v, l, r)
        elif path == "pcm16":
            oL, oR = eng.process_pcm16(quant(v), quant(l), None if r is None else quant(r))
        else:
            n = nb * B
            p = [eng.device_alloc(S * n * 4) for _ in range(5)]
            try:
                for d, a in zip(p, (v, l, r)):
                    if a is not None:
                        eng.h2d(d, a)
                eng.process_device(nb, p[0], p[1], p[2] if r is not None else None, p[3], p[4], n)
                oL, oR = np.zeros((S, n), np.float32), np.zeros((S, n), np.float32)
                eng.d2h(oL, p[3])
                eng.d2h(oR, p[4])
            finally:
                for d in p:
                    eng.device_free(d)
        self.b0 += nb
        return dict(outL=oL.copy(), outR=oR.copy(), frames=[eng.pitch_frames(s) for s in range(S)],
                    pf=[[bytes(f) for f in eng.pitch_frames(s)] for s in range(S)], vf=[eng.voc_frames(s) for s in range(S)])

    def close(self):
        self.eng.close()


def same_stream(ca, sa, cb, sb):
    if not (np.array_equal(ca["outL"][sa], cb["outL"][sb]) and np.array_equal(ca["outR"][sa], cb["outR"][sb])):
        return False
    if ca["pf"][sa] != cb["pf"][sb]:
        return False
    return all(np.array_equal(ca["vf"][sa][k], cb["vf"][sb][k]) for k in ("gated", "EeVoice", "EeSynth", "g"))


def inputs(vp, fs, S, n, first):
    return vp.synth_host(fs, S, n, flavour=0, first_stream=first)


def ref_run(fs, B, v, l, r, params):
    import oraclebind
    if refbind.available("strict"):
        return refbind.run(fs, B, v, l, synthR=r, params=params, log=True)
    return oraclebind.run(fs, B, v, l, synthR=r, params=params, log=True)


# ---------------------------------------------------------------------------------------------------------- GPU tests
# (fs, B, [(blocks, toggles)] before the move, [(blocks, toggles)] after it, mode, path)
MOVE_CONFIGS = {
    "44k1_b1024_host": (44100.0, 1024, [(19, {}), (1, dict(vocBool=0)), (2, dict(pitchBool=0))],
                        [(1, dict(pitchBool=0)), (14, {}), (9, {})], None, "host"),
    "48k_b1024_device_defined": (48000.0, 1024, [(17, {}), (2, dict(pitchBool=0))], [(3, {}), (15, {}), (8, {})], 1, "device"),
    "48k_b128_pcm16": (48000.0, 128, [(130, {}), (1, dict(vocBool=0))], [(2, dict(vocBool=0, pitchBool=0)), (40, {}), (90, {})],
                       None, "pcm16"),
}
MOVES = [(1, 4), (3, 5)]  # (source stream, slot it is loaded into)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(MOVE_CONFIGS))
def test_move_within_engine_equals_twin(vp, name):
    """Streams 1 and 3 are saved after a bypass stretch and loaded into slots 4 and 5 (whose old users differ), which from
    then on get the same input: each loaded slot equals its source, bit for bit. A run without the save / load gives the
    same streams 0..3 (saving changes nothing), and slots 4, 5 before the move."""
    fs, B, pre, post, mode, path = MOVE_CONFIGS[name]
    S = 6
    nb_pre, nb = sum(c for c, _ in pre), sum(c for c, _ in pre + post)
    n = nb * B
    V, L, R = inputs(vp, fs, S, n, 5000)
    ov, ol, orr = vp.synth_host(fs, 2, n, flavour=2, first_stream=5100)
    V[4:], L[4:], R[4:] = ov, ol, orr
    a0 = nb_pre * B
    for a, b in MOVES:
        V[b, a0:], L[b, a0:], R[b, a0:] = V[a, a0:], L[a, a0:], R[a, a0:]
    items = ITEMS + [dict(keyPitch=6, gainVoc=-10.0, gainPitch=-4.0, gainVoice=-60.0, gainSynth=-60.0)] * 2
    orders = ORDERS + [(40, 5), (48, 6)]
    pitch = PITCH + [15, 20]
    outs = {}
    for moved in (True, False):
        r = Run(vp, fs, B, S, max(c for c, _ in pre + post), items, orders, pitch, mode=mode)
        try:
            res = []
            for k, (c, q) in enumerate(pre + post):
                if k == len(pre) and moved:
                    l0 = r.eng.stats()["kernel_launches"]
                    blob = r.eng.save_streams([a for a, _ in MOVES])
                    assert r.eng.stats()["kernel_launches"] == l0
                    assert len(blob) == r.eng.snapshot_size(len(MOVES))
                    r.eng.load_streams([b for _, b in MOVES], blob)
                    r.took([b for _, b in MOVES], [items[a] for a, _ in MOVES], [orders[a] for a, _ in MOVES])
                    inf, nxt = r.eng.stream_pitch_orders()
                    for a, b in MOVES:
                        assert inf[b] == inf[a] and nxt[b] == nxt[a]
                r.toggles(**q)
                res.append(r.call(V, L, R, c, path))
            outs[moved] = res
        finally:
            r.close()
    mv, plain = outs[True], outs[False]
    for k in range(len(pre + post)):
        for s in range(4):
            assert same_stream(mv[k], s, plain[k], s), "%s: stream %d call %d changed by the save" % (name, s, k)
        for a, b in MOVES:
            if k < len(pre):
                assert same_stream(mv[k], b, plain[k], b), "%s: slot %d before the move" % (name, b)
            else:
                assert same_stream(mv[k], b, mv[k], a), "%s: slot %d != stream %d in call %d" % (name, b, a, k)
    for a, b in MOVES:  # the old user of the slot was audible: without the load the slot differs
        assert not np.array_equal(plain[len(pre)]["outL"][b], plain[len(pre)]["outL"][a])


@pytest.mark.gpu
def test_move_between_engines_and_back_matches_reference(vp):
    """Engine A runs 12 blocks, engine B 9 (a whole grid period less at 44.1 kHz / 1024): A.1 -> B.2, both run on, then
    B.2 -> A.3. Each loaded slot equals A.1 bit for bit; B's other streams are untouched; a blob saved at another phase
    (7 blocks) is refused. The stream's three pieces (A.1, B.2, A.3) match the reference on its whole input."""
    fs, B, S = 44100.0, 1024, 4
    a_pre, b_pre, mid, post = [7, 5], [9], [4, 5], [6, 8]
    nA = (sum(a_pre) + sum(mid) + sum(post)) * B
    nB = (sum(b_pre) + sum(mid) + sum(post)) * B
    VA, LA, RA = inputs(vp, fs, S, nA, 5200)
    outs = {}
    for moved in (True, False):
        VB, LB, RB = inputs(vp, fs, S, nB, 5300)
        if moved:  # B.2 gets A.1's input from the first move on
            sa, sb = sum(a_pre) * B, sum(b_pre) * B
            for D, X in ((VB, VA), (LB, LA), (RB, RA)):
                D[2, sb:] = X[1, sa:sa + nB - sb]
        A = Run(vp, fs, B, S, 9, ITEMS, ORDERS, PITCH)
        Bn = Run(vp, fs, B, S, 9, ITEMS[::-1], ORDERS[::-1], PITCH[::-1])
        try:
            ra, rb = [], []
            early = None
            for c in a_pre:
                ra.append(A.call(VA, LA, RA, c))
                if early is None:
                    early = A.eng.save_streams([1])
            for c in b_pre:
                rb.append(Bn.call(VB, LB, RB, c))
            if moved:
                with pytest.raises(vp.EngineError) as ei:
                    Bn.eng.load_streams([2], early)
                assert ei.value.code == vp.VP_E_STATE
                Bn.eng.load_streams([2], A.eng.save_streams([1]))
                Bn.took([2], [ITEMS[1]], [ORDERS[1]])
            for c in mid:
                ra.append(A.call(VA, LA, RA, c))
                rb.append(Bn.call(VB, LB, RB, c))
            if moved:
                A.eng.load_streams([3], Bn.eng.save_streams([2]))
                A.took([3], [ITEMS[1]], [ORDERS[1]])
                for D, X in ((VA, VA), (LA, LA), (RA, RA)):
                    s0 = (sum(a_pre) + sum(mid)) * B
                    D[3, s0:] = X[1, s0:]
            for c in post:
                ra.append(A.call(VA, LA, RA, c))
                rb.append(Bn.call(VB, LB, RB, c))
            outs[moved] = (ra, rb)
        finally:
            A.close()
            Bn.close()
    (ra, rb), (pa, pb) = outs[True], outs[False]
    ka, km = len(a_pre), len(mid)
    for k in range(km):
        assert same_stream(rb[1 + k], 2, ra[ka + k], 1), "B.2 != A.1 in call %d after the first move" % k
    for k in range(len(post)):
        assert same_stream(ra[ka + km + k], 3, ra[ka + km + k], 1), "A.3 != A.1 in call %d after the second move" % k
    for k in range(len(rb)):
        for s in (0, 1, 3):
            assert same_stream(rb[k], s, pb[k], s), "B.%d touched in call %d" % (s, k)
    for k in range(len(ra)):
        for s in (0, 1, 2):
            assert same_stream(ra[k], s, pa[k], s), "A.%d touched in call %d" % (s, k)
    # reference anchor: the moved stream's pieces against the reference on its whole input
    got = [ra[k]["outL"][1] for k in range(ka)] + [rb[1 + k]["outL"][2] for k in range(km)] + \
          [ra[ka + km + k]["outL"][3] for k in range(len(post))]
    frames = [f for k in range(ka) for f in ra[k]["frames"][1]] + [f for k in range(km) for f in rb[1 + k]["frames"][2]] + \
             [f for k in range(len(post)) for f in ra[ka + km + k]["frames"][3]]
    prm = refbind.default_params(lpcVoice=ORDERS[1][0], lpcSynth=ORDERS[1][1], lpcPitch=PITCH[1], **ITEMS[1])
    ref = ref_run(fs, B, VA[1], LA[1], RA[1], prm)
    got = np.concatenate(got)
    sn, mx = snr_db(ref["outL"], got), maxabs(ref["outL"], got)
    assert sn >= SNR_MIN_DB and mx <= MAXABS_MAX, "moved stream: SNR %.1f dB, max abs err %.3e" % (sn, mx)
    assert_decisions(compare_decisions(vp, oracle_decisions(ref["pitch"]), frames), "moved stream")


@pytest.mark.gpu
def test_checkpoint_into_resized_engine(vp):
    """Save the live streams of a 6-stream engine (after a pitchBool-off stretch, 48 kHz / 1024: pitch chunks straddle
    calls), prepare a 9-stream engine with a workspace small enough for several passes, load, run on: every loaded slot
    equals its source bit for bit."""
    fs, B = 48000.0, 1024
    pre, post = [(11, {}), (2, dict(pitchBool=0)), (6, {})], [(9, {}), (12, {})]
    live, slots = [0, 2, 3, 5], [7, 1, 4, 0]
    n = sum(c for c, _ in pre + post) * B
    V, L, R = inputs(vp, fs, 6, n, 5400)
    items = ITEMS + ITEMS[:2]
    orders, pitch = ORDERS + ORDERS[:2], PITCH + PITCH[:2]
    A = Run(vp, fs, B, 6, 12, items, orders, pitch)
    try:
        ra = []
        for c, q in pre:
            A.toggles(**q)
            ra.append(A.call(V, L, R, c))
        blob = A.eng.save_streams(live)
        per = A.eng.info()["workspace_bytes"] // A.eng.info()["streams_per_pass"]
        V2, L2, R2 = (np.zeros((9, n), np.float32) for _ in range(3))
        for s, t in zip(live, slots):
            V2[t], L2[t], R2[t] = V[s], L[s], R[s]
        base = [dict(keyPitch=12, gainVoc=0.0, gainPitch=0.0, gainVoice=-60.0, gainSynth=-60.0)] * 9
        C9 = Run(vp, fs, B, 9, 12, base, [(40, 5)] * 9, [15] * 9, workspace_bytes=3 * per + per // 2)
        try:
            assert -(-9 // C9.eng.info()["streams_per_pass"]) >= 3
            C9.eng.load_streams(slots, blob)
            C9.took(slots, [items[s] for s in live], [orders[s] for s in live])
            C9.b0 = A.b0
            for c, q in post:
                A.toggles(**q)
                C9.toggles(**q)
                a, b = A.call(V, L, R, c), C9.call(V2, L2, R2, c)
                for s, t in zip(live, slots):
                    assert same_stream(b, t, a, s), "slot %d != stream %d" % (t, s)
        finally:
            C9.close()
    finally:
        A.close()


@pytest.mark.gpu
def test_streaming_loads_keep_graphs_and_uniform_kernels(vp):
    """44.1 kHz / 128 streaming (BASELINE config 5's block) into a uniform 40 / 5 batch, loads between blocks:
    - a stream from a uniform batch equals its source bit for bit and adds no graph capture;
    - a stream at 40 / 5 saved from a batch whose widest rows are 64 / 8 adds no capture either: the row widths follow the
      loaded rows' own orders, so the batch stays on its tuned kernels (a stream at 40 in a batch on the generic kernels is
      matched to the reference, not bit for bit, so only the kernel choice is compared here);
    - a stream at 64 / 8 adds captures (its rows need the generic kernels) and then equals its source, whose batch is on the
      same kernels.
    The streams not loaded equal a run without loads while the batch stays uniform."""
    fs, B, S, nb, t1, t2 = 44100.0, 128, 4, 160, 70, 110
    V, L, _ = vp.synth_host(fs, S, nb * B, flavour=0, first_stream=5500, want_right=False)
    items = [dict(it, gainSynth=-60.0, gainVoice=-60.0) for it in ITEMS]

    def stream(eng, VV, LL, b):
        hv, hs, ho = eng.stream_buffers()
        hv[:] = VV[:, b * B:(b + 1) * B]
        hs[:] = LL[:, b * B:(b + 1) * B]
        eng.stream_block()
        return ho.copy()

    blobs, src = {}, {}
    for name, orders in (("uniform", [(40, 5)] * S), ("wide", [(40, 5), (64, 8), (40, 5), (40, 5)])):
        r = Run(vp, fs, B, S, 1, items, orders, [15] * S)
        try:
            o = []
            for b in range(nb):
                if b == t1:
                    blobs[name, 0] = r.eng.save_streams([0])
                if b == t2:
                    blobs[name, 1] = r.eng.save_streams([1])
                o.append(stream(r.eng, V, L, b))
            src[name] = np.concatenate(o, axis=1)
        finally:
            r.close()
    outs = {}
    for moved in (True, False):
        T = Run(vp, fs, B, S, 1, [dict(items[2])] * S, [(40, 5)] * S, [15] * S)
        VT, LT = V[[2, 3, 2, 3]].copy(), L[[2, 3, 2, 3]].copy()
        if moved:
            VT[2, t1 * B:], LT[2, t1 * B:] = V[0, t1 * B:], L[0, t1 * B:]
            VT[3, t2 * B:], LT[3, t2 * B:] = V[1, t2 * B:], L[1, t2 * B:]
        try:
            o, caps = [], []
            for b in range(nb):
                if moved and b == t1:
                    T.eng.load_streams([2], blobs["uniform", 0])
                    T.eng.load_streams([1], blobs["wide", 0])
                if moved and b == t2:
                    T.eng.load_streams([3], blobs["wide", 1])
                o.append(stream(T.eng, VT, LT, b))
                caps.append(T.eng.stream_stats()["graph_captures"])
            outs[moved] = (np.concatenate(o, axis=1), caps)
        finally:
            T.close()
    (mo, mc), (po, pc) = outs[True], outs[False]
    assert mc[:t2] == pc[:t2], "a load of narrow rows changed the captured kernels"
    assert mc[-1] > pc[-1], "a wide-order load must select the wider kernels"
    assert np.array_equal(mo[2, t1 * B:t2 * B], src["uniform"][0, t1 * B:t2 * B])
    assert np.array_equal(mo[3, t2 * B:], src["wide"][1, t2 * B:])
    assert np.array_equal(mo[0, :t2 * B], po[0, :t2 * B])
    assert np.array_equal(mo[1:3, :t1 * B], po[1:3, :t1 * B])


@pytest.mark.gpu
def test_ordering_async_reset_and_events(vp):
    """A load after an asynchronous process_device applies after it; a save waits for it; a reset pending at save time
    gives the silent record; a reset requested after a load, and an event scheduled after it, apply on top of it, while an
    event scheduled before it is dropped."""
    fs, B, S, n1, n2 = 48000.0, 1024, 4, 14, 10
    n = (n1 + n2 + 8) * B
    V, L, R = inputs(vp, fs, S, n, 5600)
    items = [dict(it, gainSynth=-60.0) for it in ITEMS]
    F = Run(vp, fs, B, S, n1, items, ORDERS, PITCH)
    E = Run(vp, fs, B, S, n1, items[::-1], ORDERS[::-1], PITCH[::-1])
    Z = Run(vp, fs, B, S, n1, items, ORDERS, PITCH)
    try:
        F.call(V, L, None, n1)
        blobF = F.eng.save_streams([0])
        p = [E.eng.device_alloc(S * n * 4) for _ in range(3)]
        try:
            VE, LE = V[::-1].copy(), L[::-1].copy()
            VE[1, n1 * B:], LE[1, n1 * B:] = V[0, n1 * B:], L[0, n1 * B:]
            E.eng.h2d(p[0], VE)
            E.eng.h2d(p[1], LE)
            at = lambda k, q: q + k * B * 4  # noqa: E731
            E.eng.process_device(10, p[0], p[1], None, p[2], None, n, sync=False)
            early = E.eng.save_streams([0, 1, 2])  # waits for the call
            E.eng.sync()
            assert early == E.eng.save_streams([0, 1, 2])
            E.eng.process_device(n1 - 10, at(10, p[0]), at(10, p[1]), None, at(10, p[2]), None, n, sync=False)
            E.eng.schedule_stream_params([(1, n1 + 2, dict(gainVoc=-30.0))])  # before the load: dropped
            E.eng.load_streams([1], blobF)  # behind the queued call
            E.eng.process_device(n2, at(n1, p[0]), at(n1, p[1]), None, at(n1, p[2]), None, n, sync=True)
            outE = np.zeros((S, n), np.float32)
            E.eng.d2h(outE, p[2])
        finally:
            for d in p:
                E.eng.device_free(d)
        f2 = F.call(V, L, None, n2)
        assert np.array_equal(outE[1, n1 * B:(n1 + n2) * B], f2["outL"][0]), "the load did not apply after the queued call"
        assert E.eng.stream_params(1, 1)[0] == vp.stream_params(**items[0]).as_dict(), "an event from before the load survived"
        # a pending reset: the saved raw state is the silent state of a stream that processed nothing
        rec = E.eng.snapshot_size(1) - vp.VP_SNAPSHOT_HEADER_BYTES
        raw = slice(vp.VP_SNAPSHOT_HEADER_BYTES + vp.VP_SNAPSHOT_RECORD_BYTES, vp.VP_SNAPSHOT_HEADER_BYTES + rec)
        silent = Z.eng.save_streams([3])[raw]
        assert E.eng.save_streams([3])[raw] != silent
        E.eng.reset_streams([3])
        assert E.eng.save_streams([3])[raw] == silent
        # reset / event after a load apply on top: F.2 and F.3 end up as F.1 reset, with F.1's values and a later gain event
        F.eng.load_streams([2, 3], F.eng.save_streams([0, 1]))
        F.took([2, 3], [items[0], items[1]], [ORDERS[0], ORDERS[1]])
        F.eng.reset_streams([1, 3])
        ev = [(s, n1 + n2 + 3, dict(gainVoc=-9.0)) for s in (0, 2)]
        F.eng.schedule_stream_params(ev)
        W = dict(V=V.copy(), L=L.copy())
        for D in (W["V"], W["L"]):
            D[2], D[3] = D[0], D[1]
        f3 = F.call(W["V"], W["L"], None, 8)
        assert same_stream(f3, 2, f3, 0), "event after the load"
        assert same_stream(f3, 3, f3, 1), "reset after the load"
    finally:
        F.close()
        E.close()
        Z.close()


@pytest.mark.gpu
def test_rejected_blobs_change_nothing(vp):
    """Wrong magic, version, layout (another block size, reservation, window), another grid phase, a flipped byte, a mark
    count above VP_SLOTS with a repaired checksum, a short buffer, a duplicate slot: each returns its code, launches nothing,
    and the engine continues bit for bit as one that never saw the call."""
    fs, B, S = 44100.0, 1024, 3
    V, L, R = inputs(vp, fs, S, 20 * B, 5700)
    items, orders, pitch = ITEMS[:3], ORDERS[:3], PITCH[:3]
    plain = Run(vp, fs, B, S, 8, items, orders, pitch)
    E = Run(vp, fs, B, S, 8, items, orders, pitch)
    others = []
    try:
        p0, e0 = plain.call(V, L, R, 6), E.call(V, L, R, 6)
        good = E.eng.save_streams([0])
        rec_bytes = len(good) - vp.VP_SNAPSHOT_HEADER_BYTES
        units, seg = units_per_stream(E.eng.sizes, B, E.eng.info()["history_samples"], 64, 8)
        assert rec_bytes == vp.VP_SNAPSHOT_RECORD_BYTES + 16 * units
        assert E.eng.snapshot_size(3) == vp.VP_SNAPSHOT_HEADER_BYTES + 3 * rec_bytes
        bad = {}
        b = bytearray(good); b[0] ^= 1; bad["magic"] = (bytes(b), vp.VP_E_ARG)
        b = bytearray(good); b[4] = 7; bad["version"] = (bytes(b), vp.VP_E_ARG)
        b = bytearray(good); b[-100] ^= 0x40; bad["flipped byte"] = (bytes(b), vp.VP_E_ARG)
        b = bytearray(good); b[20] ^= 0x01; bad["flipped header byte"] = (bytes(b), vp.VP_E_ARG)
        marks = vp.VP_SNAPSHOT_HEADER_BYTES + vp.VP_SNAPSHOT_RECORD_BYTES + seg["marks"]
        b = bytearray(good); b[marks + 24:marks + 28] = (40).to_bytes(4, "little")  # VPMarkState.nAn
        bad["nAn > VP_SLOTS"] = (fix_record_checksum(bytes(b), 0, rec_bytes, vp), vp.VP_E_RANGE)
        b = bytearray(good); b[marks + 8:marks + 12] = (100000).to_bytes(4, "little")  # VPMarkState.prevVoicedPeriod
        bad["period > tauMax"] = (fix_record_checksum(bytes(b), 0, rec_bytes, vp), vp.VP_E_RANGE)
        bad["short buffer"] = (good[:-16], vp.VP_E_ARG)
        for what, kw in (("block size", dict(block=128)), ("reservation", dict(reserve_orders=(48, 8))),
                         ("window", dict(window=vp.VP_WINDOW_HANN))):
            o = vp.Engine(fs, kw.get("block", B), S, 8, reserve_orders=kw.get("reserve_orders", RESERVE),
                          reserve_pitch_order=RESERVE_P, window=kw.get("window", vp.VP_WINDOW_SINE))
            others.append(o)
            bad["layout: " + what] = (o.save_streams([0]), vp.VP_E_STATE)
        ph = Run(vp, fs, B, S, 8, items, orders, pitch)
        others.append(ph.eng)
        ph.call(V, L, R, 7)
        bad["grid phase"] = (ph.eng.save_streams([0]), vp.VP_E_STATE)
        l0 = E.eng.stats()["kernel_launches"]
        for what, (blob, code) in bad.items():
            with pytest.raises(vp.EngineError) as ei:
                E.eng.load_streams([1], blob)
            assert ei.value.code == code, "%s: code %d" % (what, ei.value.code)
        arr = (C.c_int * 2)(1, 1)
        two = E.eng.save_streams([0, 0])
        assert E.eng.lib.vp_engine_load_streams(E.eng.h, arr, 2, two, len(two)) == vp.VP_E_ARG
        assert E.eng.lib.vp_engine_load_streams(E.eng.h, arr, 1, two, len(two)) == vp.VP_E_ARG  # count != records
        assert E.eng.stats()["kernel_launches"] == l0
        for k in range(2):
            a, b2 = plain.call(V, L, R, 7), E.call(V, L, R, 7)
            for s in range(S):
                assert same_stream(a, s, b2, s), "stream %d call %d after the rejected loads" % (s, k)
        # before prepare
        lib = vp.load_library()
        h = C.c_void_p()
        assert lib.vp_engine_create(C.byref(h), 0) == vp.VP_OK
        try:
            n = C.c_size_t(0)
            assert lib.vp_engine_snapshot_size(h, 1, C.byref(n)) == vp.VP_E_STATE
            one = (C.c_int * 1)(0)
            assert lib.vp_engine_save_streams(h, one, 1, C.create_string_buffer(len(good)), len(good)) == vp.VP_E_STATE
            assert lib.vp_engine_load_streams(h, one, 1, good, len(good)) == vp.VP_E_STATE
        finally:
            lib.vp_engine_destroy(h)
        # a save with a bad list or a short buffer
        for lst, nbytes in (([3], len(good)), ([-1], len(good)), ([0], len(good) - 1)):
            arr1 = (C.c_int * 1)(*lst)
            assert E.eng.lib.vp_engine_save_streams(E.eng.h, arr1, 1, C.create_string_buffer(len(good)), nbytes) == vp.VP_E_ARG
    finally:
        plain.close()
        E.close()
        for o in others:
            o.close()
