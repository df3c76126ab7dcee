#!/usr/bin/env python3
"""Cost of block-accurate per-stream automation (vp_engine_schedule_stream_params), in one run:

  device:    the default bench workload (chain48: 2048 streams x 60 s @ 48 kHz, block 1024, full chain, device-resident) in
             three layouts, alternating round by round in one engine: (a) no events; (b) 8 events per stream at random
             blocks (key, gainVoc, gainPitch), dry paths off; (c) as (b) plus dry-voice on / off events on half the streams.
             Step = vp_engine_reset, the starting values, the schedule, then one process call over the whole batch; the call
             is timed with CUDA events on the engine's stream (what it issues: table upload, expansion kernel, passes).
  cut:       the alternative to (b) without the feature: the call cut at the union of all event blocks, with
             vp_engine_set_stream_params between the parts (2048 streams x 10 s), against one scheduled call of the same.
  streaming: BASELINE config 5 (4096 streams, block 128 at 44.1 kHz) with 0, 64 and 4096 events per block; per block the host
             clock from the schedule request to the return of vp_engine_stream_block; p50 / p99 against the 2.90 ms period.
  parity:    16 streams of (b) and of (c) against the reference run with each stream's own schedule.

The card's name, power limit and clocks are read in the same run.

    python tools/stream_schedule_bench.py [--out FILE]

Prints one JSON line (and writes it to --out). Writes nothing else."""
import argparse
import ctypes as C
import json
import os
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from stream_params_bench import card_info  # noqa: E402  (tools/ is this script's directory)

FIELDS = ("gainPitch", "gainVoice", "gainSynth", "gainVoc", "keyPitch")


def layout(S, nb, kind, seed=11):
    """(starting values, [(stream, block, values)]) of layout a / b / c."""
    rng = np.random.RandomState(seed)
    base = [dict(keyPitch=s % 13, gainVoc=0.0, gainPitch=0.0, gainVoice=-60.0, gainSynth=-60.0) for s in range(S)]
    if kind == "a":
        return base, []
    ev = []
    for s in range(S):
        cur = dict(base[s])
        blocks = sorted(rng.choice(np.arange(1, nb), 8, replace=False))
        for k, b in enumerate(blocks):
            cur = dict(cur, keyPitch=int(rng.randint(0, 13)), gainVoc=float(rng.uniform(-20.0, 6.0)),
                       gainPitch=float(rng.uniform(-20.0, 6.0)))
            if kind == "c" and s % 2 == 0:
                cur["gainVoice"] = float(rng.uniform(-30.0, 0.0)) if k % 2 == 0 else -60.0
            ev.append((s, int(b), dict(cur)))
    return base, ev


def event_array(vp, events):
    arr = (vp.StreamEvent * max(len(events), 1))()
    for k, (s, b, v) in enumerate(events):
        arr[k].stream, arr[k].block = s, b
        for f in FIELDS:
            setattr(arr[k].p, f, v[f])
    return arr


def device_leg(vp, steps, rounds, dev, seconds=60.0):
    fs, B, S = 48000.0, 1024, 2048
    n = int(fs * seconds) // B * B
    nb = n // B
    eng = vp.Engine(fs, B, S, nb, device=dev)
    bufs = [eng.device_alloc(S * n * 4) for _ in range(3)]
    dv, dl, do = bufs
    eng.synth_device(0, 0, S, n, n, dv, dl, None)
    kinds = ("a", "b", "c")
    lays = {k: layout(S, nb, k) for k in kinds}
    arrs = {k: event_array(vp, lays[k][1]) for k in kinds}
    times = {k: [] for k in kinds}
    launches = {}

    def step(k):
        eng.reset()
        eng.set_stream_params(0, lays[k][0])
        if lays[k][1]:
            eng._check(eng.lib.vp_engine_schedule_stream_params(eng.h, arrs[k], len(lays[k][1])))
        eng.timer_record(0)
        l0 = eng.stats()["kernel_launches"]
        eng.process_device(nb, dv, dl, None, do, None, n, sync=False)
        launches[k] = eng.stats()["kernel_launches"] - l0
        eng.timer_record(1)
        return eng.timer_elapsed_ms(0, 1)
    try:
        for _ in range(rounds):
            for k in kinds:
                step(k)  # warm-up step of this layout
                times[k].append(float(np.median([step(k) for _ in range(steps)])))
        sp = eng.info()["streams_per_pass"]
        par = {}
        for k in ("b", "c"):
            step(k)
            eng.sync()
            par[k] = parity(vp, eng, fs, B, S, n, dv, dl, do, lays[k])
    finally:
        for p in bufs:
            eng.device_free(p)
        eng.close()
    res = {"workload": "chain48: %d streams x %.1f s @ 48 kHz, block 1024, device-resident" % (S, n / fs), "streams_per_pass": sp,
           "steps_per_round": steps, "rounds": rounds, "timer": "CUDA events on the engine's stream around each process call",
           "events": {k: len(lays[k][1]) for k in kinds}, "launches_per_call": launches, "layouts": {}, "parity": par}
    base = float(np.median(times["a"]))
    for k, t in times.items():
        med = float(np.median(t))
        res["layouts"][k] = {"ms_per_call_median": med, "ms_per_call_rounds": t, "spread_ms": float(max(t) - min(t)),
                             "delta_vs_a_ms": med - base, "delta_vs_a_pct": 100.0 * (med - base) / base}
    return res


def parity(vp, eng, fs, B, S, n, dv, dl, do, lay, want=16):
    import oraclebind
    import refbind
    from common import MAXABS_MAX, SNR_MIN_DB, compare_decisions, maxabs, oracle_decisions, snr_db
    base, events = lay
    picks = sorted({int(round(x)) for x in np.linspace(0, S - 1, want)})
    use_ref = refbind.available("strict")
    ins, outs = [], {}
    for s in picks:
        v, l, o = np.zeros(n, np.float32), np.zeros(n, np.float32), np.zeros(n, np.float32)
        for arr, p in ((v, dv), (l, dl), (o, do)):
            eng._check(eng.lib.vp_memcpy_d2h(eng.h, arr.ctypes.data, C.c_void_p(p + s * n * 4), n * 4))
        sched = [(b, refbind.default_params(**x)) for t, b, x in events if t == s]
        ins.append((v, l, refbind.default_params(**base[s]), sched))
        outs[s] = o

    def one(job):
        v, l, prm, sched = job
        mod = refbind if use_ref else oraclebind
        return mod.run(fs, B, v, l, synthR=None, params=prm, log=True, schedule=sched)
    if not use_ref:
        oraclebind.load()
    t0 = time.time()
    with ThreadPoolExecutor(max_workers=max(1, len(os.sched_getaffinity(0)))) as ex:
        refs = list(ex.map(one, ins))
    cpu_s = time.time() - t0
    worst_snr, worst_abs, tot, chk, bad = 1e9, 0.0, 0, 0, 0
    for s, r in zip(picks, refs):
        worst_snr = min(worst_snr, snr_db(r["outL"], outs[s]))
        worst_abs = max(worst_abs, maxabs(r["outL"], outs[s]))
        dec = compare_decisions(vp, oracle_decisions(r["pitch"]), eng.pitch_frames(s))
        tot += dec.n; chk += dec.checked; bad += dec.bad
    ok = worst_snr >= SNR_MIN_DB and worst_abs <= MAXABS_MAX and bad == 0 and chk >= 0.98 * tot
    return {"streams": len(picks), "seconds": n / fs, "reference": "reference" if use_ref else "port", "worst_snr_db": worst_snr,
            "worst_maxabs": worst_abs, "frames": tot, "frames_compared": chk, "mismatches": bad, "cpu_seconds": cpu_s, "ok": bool(ok)}


def cut_leg(vp, dev, seconds=10.0):
    """Layout (b) at 2048 x 10 s: one scheduled call against the call cut at every event block."""
    fs, B, S = 48000.0, 1024, 2048
    n = int(fs * seconds) // B * B
    nb = n // B
    base, events = layout(S, nb, "b")
    eng = vp.Engine(fs, B, S, nb, device=dev)
    bufs = [eng.device_alloc(S * n * 4) for _ in range(3)]
    dv, dl, do = bufs
    eng.synth_device(0, 0, S, n, n, dv, dl, None)
    arr = event_array(vp, events)
    by = {}
    for s, b, v in events:
        by.setdefault(b, []).append((s, v))
    cuts = sorted({0, nb} | set(by))
    res = {}
    try:
        for rep in range(2):  # the first repetition warms up every call length
            eng.reset()
            eng.set_stream_params(0, base)
            eng._check(eng.lib.vp_engine_schedule_stream_params(eng.h, arr, len(events)))
            eng.sync()
            t0 = time.perf_counter()
            eng.process_device(nb, dv, dl, None, do, None, n, sync=True)
            one = time.perf_counter() - t0
            eng.reset()
            eng.set_stream_params(0, base)
            eng.sync()
            t0 = time.perf_counter()
            for a, b in zip(cuts, cuts[1:]):
                for s, v in by.get(a, []):
                    eng.set_stream_params(s, [v])
                eng.process_device(b - a, dv + a * B * 4, dl + a * B * 4, None, do + a * B * 4, None, n, sync=False)
            eng.sync()
            cut = time.perf_counter() - t0
            res = {"one_call_ms": one * 1e3, "cut_calls": len(cuts) - 1, "cut_ms": cut * 1e3, "ratio": cut / one}
    finally:
        for p in bufs:
            eng.device_free(p)
        eng.close()
    res.update({"workload": "layout b at %d streams x %.1f s @ 48 kHz, block 1024, device-resident" % (S, n / fs),
                "events": len(events), "timer": "host clock around the call(s), ending in a device synchronise"})
    return res


def streaming_leg(vp, blocks, rounds, dev):
    fs, Bs, S = 44100.0, 128, 4096
    pool = 64
    v, l, _ = vp.synth_host(fs, 256, pool * Bs, flavour=0, first_stream=0, want_right=False)
    V, L = np.tile(v, (S // 256, 1)), np.tile(l, (S // 256, 1))
    eng = vp.Engine(fs, Bs, S, 1, device=dev)
    counts = (0, 64, 4096)
    rng = np.random.RandomState(3)
    arrs = {}
    for k in counts:  # values prepared once; the block field is set per block through a numpy view
        a = (vp.StreamEvent * max(k, 1))()
        for i in range(k):
            a[i].stream = int(i * S // k)
            a[i].p.keyPitch, a[i].p.gainVoc, a[i].p.gainPitch = int(rng.randint(0, 13)), float(rng.uniform(-20, 6)), float(rng.uniform(-20, 6))
            a[i].p.gainVoice = a[i].p.gainSynth = -60.0
        view = np.frombuffer(a, dtype=np.dtype({"names": ["block"], "formats": ["<i8"], "offsets": [8], "itemsize": 40}))
        arrs[k] = (a, view)
    lat = {k: [] for k in counts}
    try:
        hv, hs, _ = eng.stream_buffers()
        b = 0

        def block(k):
            nonlocal b
            x = slice((b % pool) * Bs, (b % pool + 1) * Bs)
            hv[:] = V[:, x]
            hs[:] = L[:, x]
            t0 = time.perf_counter()
            if k:
                a, view = arrs[k]
                view["block"] = b
                eng._check(eng.lib.vp_engine_schedule_stream_params(eng.h, a, k))
            eng.stream_block()
            t = time.perf_counter() - t0
            b += 1
            return t
        for _ in range(300):
            block(0)
        cap0 = eng.stream_stats()["graph_captures"]
        for _ in range(rounds):
            for k in counts:
                for _ in range(blocks):
                    lat[k].append(block(k))
        captures = eng.stream_stats()["graph_captures"] - cap0
    finally:
        eng.close()
    period = Bs / fs * 1e3
    res = {"workload": "BASELINE config 5: %d streams, block %d @ 44.1 kHz, CUDA graph per block phase" % (S, Bs),
           "block_period_ms": period, "blocks_per_config": blocks * rounds, "rounds": rounds,
           "timer": "host clock from the schedule request to the return of vp_engine_stream_block",
           "graph_captures_while_timed": captures, "events_per_block": {}}
    for k, t in lat.items():
        a = np.array(t) * 1e3
        res["events_per_block"][str(k)] = {"p50_ms": float(np.percentile(a, 50)), "p99_ms": float(np.percentile(a, 99)),
                                           "max_ms": float(a.max()), "p99_within_period": bool(np.percentile(a, 99) < period)}
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=60.0)
    ap.add_argument("--stream-blocks", type=int, default=500, help="timed blocks per configuration and round")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import vocoderproject_b200 as vp
    res = {"tool": "stream_schedule_bench", "card": card_info(args.device)}
    res["device"] = device_leg(vp, args.steps, args.rounds, args.device, args.seconds)
    res["cut"] = cut_leg(vp, args.device)
    res["streaming"] = streaming_leg(vp, args.stream_blocks, args.rounds, args.device)
    res["card_after"] = card_info(args.device)
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
