#!/usr/bin/env python3
"""Cost of per-stream vocoder orders (vp_engine_set_stream_orders / vp_engine_schedule_stream_orders), in one run, on the
default bench workload (chain48: 2048 streams x 60 s @ 48 kHz, block 1024, full chain, device-resident):

  leg 1, one engine prepared as bench.py prepares it, layouts alternating round by round:
    (a) uniform defaults (lpcVoice 40, lpcSynth 5 on every stream);
    (b) random per-stream orders, lpcVoice 2..40, lpcSynth 2..5;
    (c) (b) plus one scheduled order change per stream at a random block inside the call.
  leg 2, one engine with vp_engine_reserve_orders(64, 5) (its rows are 65 wide: the workspace differs from leg 1):
    (a') as (a);  (d) as (a) with a single stream at lpcVoice 64 (the whole call then runs the generic kernels).

Step = vp_engine_reset, the layout's orders (and schedule), then one process call over the whole batch, timed with CUDA
events on the engine's stream. The engine's stage timers are on (VP_STAGE_TIMING=1) in every layout, so that the
voc_levinson stage (vp_engine_last_timing) is read from the same calls. Per layout: ms per call (median over rounds and
their spread), stage times, kernel launches per call, and parity of 16 streams against the reference run at each stream's
own orders (and schedule). The card's name, power limit and clocks are read in the same run.

    python tools/stream_orders_bench.py [--out FILE]

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


def layout(S, nb, kind, seed=13):
    """(per-stream orders, [(stream, block, orders)]) of layout a / b / c / d."""
    rng = np.random.RandomState(seed)
    if kind == "a":
        return [(40, 5)] * S, []
    if kind == "d":
        return [(40, 5)] * (S // 2) + [(64, 5)] + [(40, 5)] * (S - S // 2 - 1), []
    base = [(int(rng.randint(2, 41)), int(rng.randint(2, 6))) for _ in range(S)]
    ev = []
    if kind == "c":
        ev = [(s, int(rng.randint(1, nb)), (int(rng.randint(2, 41)), int(rng.randint(2, 6)))) for s in range(S)]
    return base, ev


def order_arrays(vp, base, events):
    o = (vp.StreamOrders * len(base))()
    for k, (v, s) in enumerate(base):
        o[k].lpcVoice, o[k].lpcSynth = v, s
    ev = (vp.StreamOrderEvent * max(len(events), 1))()
    for k, (s, b, (ov, os_)) in enumerate(events):
        ev[k].stream, ev[k].block, ev[k].o.lpcVoice, ev[k].o.lpcSynth = s, b, ov, os_
    return o, ev


def leg(vp, kinds, steps, rounds, dev, seconds, reserve=None):
    fs, B, S = 48000.0, 1024, 2048
    n = int(fs * seconds) // B * B
    nb = n // B
    eng = vp.Engine(fs, B, S, nb, device=dev, reserve_orders=reserve)
    bufs = [eng.device_alloc(S * n * 4) for _ in range(3)]
    dv, dl, do = bufs
    eng.synth_device(0, 0, S, n, n, dv, dl, None)
    lays = {k: layout(S, nb, k) for k in kinds}
    arrs = {k: order_arrays(vp, *lays[k]) for k in kinds}
    times = {k: [] for k in kinds}
    stages = {k: [] for k in kinds}
    launches = {}

    def step(k):
        eng.reset()
        o, ev = arrs[k]
        eng._check(eng.lib.vp_engine_set_stream_orders(eng.h, 0, S, o))
        if lays[k][1]:
            eng._check(eng.lib.vp_engine_schedule_stream_orders(eng.h, ev, len(lays[k][1])))
        eng.timer_record(0)
        l0 = eng.stats()["kernel_launches"]
        eng.process_device(nb, dv, dl, None, do, None, n, sync=False)
        launches[k] = eng.stats()["kernel_launches"] - l0
        eng.timer_record(1)
        ms = eng.timer_elapsed_ms(0, 1)
        return ms, eng.last_timing()[1]
    try:
        for _ in range(rounds):
            for k in kinds:
                step(k)  # warm-up step of this layout
                got = [step(k) for _ in range(steps)]
                times[k].append(float(np.median([g[0] for g in got])))
                stages[k].append({st: float(np.median([g[1][st] for g in got])) for st in got[0][1] if st})
        sp = eng.info()["streams_per_pass"]
        par = {}
        for k in kinds:
            step(k)
            eng.sync()
            par[k] = parity(vp, eng, fs, B, S, n, dv, dl, do, lays[k])
    finally:
        for p in bufs:
            eng.device_free(p)
        eng.close()
    res = {"workload": "chain48: %d streams x %.1f s @ 48 kHz, block 1024, device-resident" % (S, n / fs),
           "reserve_orders": reserve, "streams_per_pass": sp, "steps_per_round": steps, "rounds": rounds,
           "timer": "CUDA events on the engine's stream around each process call (stage timers on)",
           "launches_per_call": launches, "layouts": {}, "parity": par}
    base = float(np.median(times[kinds[0]]))
    for k, t in times.items():
        med = float(np.median(t))
        st = {name: float(np.median([r[name] for r in stages[k]])) for name in stages[k][0]}
        res["layouts"][k] = {"ms_per_call_median": med, "ms_per_call_rounds": t, "spread_ms": float(max(t) - min(t)),
                             "delta_vs_%s_ms" % kinds[0]: med - base, "delta_vs_%s_pct" % kinds[0]: 100.0 * (med - base) / base,
                             "voc_levinson_ms_rounds": [r["voc_levinson"] for r in stages[k]], "stage_ms_median": st}
    return res


def parity(vp, eng, fs, B, S, n, dv, dl, do, lay, want=16):
    import oraclebind
    import refbind
    from common import MAXABS_MAX, SNR_MIN_DB, compare_decisions, maxabs, oracle_decisions, snr_db
    base, events = lay
    picks = sorted({int(round(x)) for x in np.linspace(0, S - 1, want)} | {s for s, o in enumerate(base) if o[0] > 40})
    use_ref = refbind.available("strict")
    ins, outs = [], {}
    for s in picks:
        v, l, o = np.zeros(n, np.float32), np.zeros(n, np.float32), np.zeros(n, np.float32)
        for arr, p in ((v, dv), (l, dl), (o, do)):
            eng._check(eng.lib.vp_memcpy_d2h(eng.h, arr.ctypes.data, C.c_void_p(p + s * n * 4), n * 4))
        sched = [(b, refbind.default_params(lpcVoice=x[0], lpcSynth=x[1])) for t, b, x in events if t == s]
        ins.append((v, l, refbind.default_params(lpcVoice=base[s][0], lpcSynth=base[s][1]), sched))
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


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=60.0)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    os.environ["VP_STAGE_TIMING"] = "1"  # read by vp_engine_create
    import vocoderproject_b200 as vp
    res = {"tool": "stream_orders_bench", "card": card_info(args.device)}
    res["leg1"] = leg(vp, ("a", "b", "c"), args.steps, args.rounds, args.device, args.seconds)
    res["leg2"] = leg(vp, ("a", "d"), args.steps, args.rounds, args.device, args.seconds, reserve=(64, 5))
    res["card_after"] = card_info(args.device)
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
