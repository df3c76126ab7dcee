#!/usr/bin/env python3
"""Cost of per-stream parameters: the default bench workload (chain48: 2048 streams x 60 s @ 48 kHz, block 1024, full
chain, device-resident) timed with three parameter layouts in one engine, alternating round by round:

  (a) uniform parameters (every stream the plug-in's defaults, what bench.py runs),
  (b) 13 keys and random gains across the streams, dry paths off,
  (c) as (b) with the dry voice on for half of the streams (the general mix kernel instead of the 128-bit one).

Switching layouts is vp_engine_set_stream_params only (table data, no re-prepare). Step = reset + one process call over
the whole batch, timed with CUDA events on the engine's stream. After the last timed step of (b) and (c) a spread of >= 16
streams (incl. the first and last stream of every pass) is compared, for the full 60 s, with the reference run with each
stream's own parameters, as bench.py's parity object does. The card's name and power limit are read in the same run.

    python tools/stream_params_bench.py [--steps 5] [--rounds 3] [--streams 2048] [--out FILE]

Prints one JSON line (and writes it to --out). Writes nothing else."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card_info(dev):
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=60).stdout.strip().split(", ")
        return {"name": out[0], "power_limit_w": float(out[1]), "sm_max_mhz": float(out[2])}
    except Exception as ex:  # the timing stands without it, but says so
        return {"error": "nvidia-smi: %r" % (ex,)}


def layouts(S, seed=7):
    rng = np.random.RandomState(seed)
    b = [dict(keyPitch=s % 13, gainVoc=float(rng.uniform(-20.0, 6.0)), gainPitch=float(rng.uniform(-20.0, 6.0)),
              gainVoice=-60.0, gainSynth=-60.0) for s in range(S)]
    c = [dict(it, gainVoice=float(rng.uniform(-30.0, 0.0)) if s % 2 == 0 else -60.0) for s, it in enumerate(b)]
    return {"a_uniform": None, "b_keys_gains": b, "c_keys_gains_half_dry_voice": c}


def parity(vp, eng, fs, B, S, n, dv, dl, do, items, want=16):
    from common import MAXABS_MAX, SNR_MIN_DB, compare_decisions, maxabs, oracle_decisions, reference_runs, snr_db
    Sc = eng.info()["streams_per_pass"]
    picks = set()
    for p0 in range(0, S, Sc):
        picks |= {p0, min(p0 + Sc, S) - 1}
    want = max(want, len(picks))
    for x in np.linspace(0, S - 1, want):
        if len(picks) >= want:
            break
        picks.add(int(round(x)))
    picks = sorted(picks)
    ins, outs = [], {}
    for s in picks:
        v, l, o = np.zeros(n, np.float32), np.zeros(n, np.float32), np.zeros(n, np.float32)
        for arr, base in ((v, dv), (l, dl), (o, do)):
            eng._check(eng.lib.vp_memcpy_d2h(eng.h, arr.ctypes.data, C.c_void_p(base + s * n * 4), n * 4))
        ins.append((fs, B, v, l, None, items[s]))
        outs[s] = o
    t0 = time.time()
    refs, kind = reference_runs(ins)
    cpu_s = time.time() - t0
    worst_snr, worst_abs, tot, chk, flg, bad = 1e9, 0.0, 0, 0, 0, 0
    for s, r in zip(picks, refs):
        worst_snr = min(worst_snr, snr_db(r["outL"], outs[s]))
        worst_abs = max(worst_abs, maxabs(r["outL"], outs[s]))
        dec = compare_decisions(vp, oracle_decisions(r["pitch"]), eng.pitch_frames(s))
        tot += dec.n; chk += dec.checked; flg += dec.flagged; bad += dec.bad
    ok = worst_snr >= SNR_MIN_DB and worst_abs <= MAXABS_MAX and bad == 0 and chk >= 0.98 * tot
    return {"streams": len(picks), "streams_checked": picks, "seconds": n / fs, "reference": kind, "worst_snr_db": worst_snr,
            "worst_maxabs": worst_abs, "frames": tot, "frames_compared": chk, "frames_flagged": flg, "mismatches": bad,
            "keys": sorted({items[s]["keyPitch"] for s in picks}), "dry_voice_streams": sum(items[s]["gainVoice"] > -59.0 for s in picks),
            "cpu_seconds": cpu_s, "ok": bool(ok)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--streams", type=int, default=2048)
    ap.add_argument("--seconds", type=float, default=60.0)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import vocoderproject_b200 as vp
    fs, B, S = 48000.0, 1024, args.streams
    n = int(fs * args.seconds) // B * B
    nb = n // B
    card = card_info(args.device)
    eng = vp.Engine(fs, B, S, nb, device=args.device)
    dv, dl, do = (eng.device_alloc(S * n * 4) for _ in range(3))
    eng.synth_device(0, 0, S, n, n, dv, dl, None)
    uniform = [vp.stream_params().as_dict()] * S
    lay = layouts(S)
    times = {k: [] for k in lay}
    par = {}
    for r in range(args.rounds):
        for name, items in lay.items():
            eng.set_stream_params(0, items if items is not None else uniform)
            eng.reset()
            eng.process_device(nb, dv, dl, None, do, None, n, sync=False)  # warm-up step of this layout
            eng.sync()
            eng.timer_record(0)
            for _ in range(args.steps):
                eng.reset()
                eng.process_device(nb, dv, dl, None, do, None, n, sync=False)
            eng.timer_record(1)
            eng.sync()
            times[name].append(eng.timer_elapsed_ms(0, 1) / args.steps)
            if r == args.rounds - 1 and items is not None:
                par[name] = parity(vp, eng, fs, B, S, n, dv, dl, do, items)
    for p in (dv, dl, do):
        eng.device_free(p)
    info = eng.info()
    eng.close()
    res = {"tool": "stream_params_bench", "card": card,
           "workload": "chain48: %d streams x %.1f s @ 48 kHz, block 1024, full chain, device-resident" % (S, n / fs),
           "steps_per_round": args.steps, "rounds": args.rounds, "streams_per_pass": info["streams_per_pass"],
           "timer": "CUDA events on the engine's stream around each round's steps (reset + one process call per step)",
           "configs": {}}
    for name, t in times.items():
        med = float(np.median(t))
        res["configs"][name] = {"ms_per_step_median": med, "ms_per_step_rounds": t, "spread_ms": float(max(t) - min(t)),
                                "x_realtime": S * n / fs / (med * 1e-3)}
    a = res["configs"]["a_uniform"]["ms_per_step_median"]
    for name in res["configs"]:
        res["configs"][name]["vs_uniform"] = res["configs"][name]["ms_per_step_median"] / a
    res["parity"] = par
    res["ok"] = all(p["ok"] for p in par.values())
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0 if res["ok"] else 1


if __name__ == "__main__":
    sys.exit(main())
