#!/usr/bin/env python3
"""Cost of per-stream pitch-corrector orders (vp_engine_set_stream_pitch_orders), in one run, on the default bench workload
(chain48: 2048 streams x 60 s @ 48 kHz, block 1024, full chain, device-resident):

  leg 1, one engine prepared as bench.py prepares it (lpcPitch 15, no reservation), layouts alternating round by round:
    (a) uniform 15 on every stream (the call bench.py makes);
    (b) lpcPitch spread over 2..15, both ends included (rows padded to 16: the P = 15 residual path, per-frame Levinson
        and all-pole forms);
    (u9) uniform 9 on every stream: the kernels an engine prepared at 9 runs (generic Levinson, residual and direct-form
        all-pole filter), which is what most streams of (b) run as well.
  leg 2, one engine with vp_engine_reserve_pitch_order(100) (its pitch rows are 101 wide: the workspace differs from leg 1):
    (a') as (a);  (c) lpcPitch spread over 2..100 (rows 101 wide, generic residual, per-frame Levinson and all-pole forms);
    (u51) uniform 51, the middle of (c)'s orders, on the generic kernels.

Step = vp_engine_reset, the layout's orders, then one process call over the whole batch, timed with CUDA events on the
engine's stream. The engine's stage timers are on (VP_STAGE_TIMING=1) in every layout, so the pitch stages (pitch_lpc =
autocorrelation + Levinson, pitch_psola, pitch_iir) are read from the same calls. Per layout: ms per call (median over
rounds and their spread), stage times and kernel launches per call. The card's name, power limit and clocks are read in
the same run. Bit parity of mixed layouts against solo engines is what tests/test_stream_pitch_orders.py checks.

    python tools/stream_pitch_orders_bench.py [--out FILE]

Prints one JSON line (and writes it to --out). Writes nothing else."""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from stream_params_bench import card_info  # noqa: E402  (tools/ is this script's directory)

PITCH_STAGES = ("pitch_lpc", "pitch_psola", "pitch_iir")


def layout(S, kind):
    if kind in ("a", "a'"):
        return [15] * S
    if kind.startswith("u"):
        return [int(kind[1:])] * S
    hi = 15 if kind == "b" else 100
    return [int(x) for x in np.linspace(2, hi, S).round()]


def leg(vp, kinds, steps, rounds, dev, seconds, reserve=None):
    fs, B, S = 48000.0, 1024, 2048
    n = int(fs * seconds) // B * B
    nb = n // B
    eng = vp.Engine(fs, B, S, nb, device=dev, reserve_pitch_order=reserve)
    bufs = [eng.device_alloc(S * n * 4) for _ in range(3)]
    dv, dl, do = bufs
    eng.synth_device(0, 0, S, n, n, dv, dl, None)
    arrs = {k: (C.c_int * S)(*layout(S, k)) for k in kinds}
    times = {k: [] for k in kinds}
    stages = {k: [] for k in kinds}
    launches = {}

    def step(k):
        eng._check(eng.lib.vp_engine_set_stream_pitch_orders(eng.h, 0, S, arrs[k]))
        eng.reset()  # every stream starts with the layout's order
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
        info = eng.info()
    finally:
        for p in bufs:
            eng.device_free(p)
        eng.close()
    res = {"workload": "chain48: %d streams x %.1f s @ 48 kHz, block 1024, device-resident" % (S, n / fs),
           "reserve_pitch_order": reserve, "streams_per_pass": info["streams_per_pass"], "workspace_bytes": info["workspace_bytes"],
           "steps_per_round": steps, "rounds": rounds,
           "timer": "CUDA events on the engine's stream around each process call (stage timers on)",
           "launches_per_call": launches, "layouts": {}}
    base = float(np.median(times[kinds[0]]))
    for k, t in times.items():
        med = float(np.median(t))
        st = {name: float(np.median([r[name] for r in stages[k]])) for name in stages[k][0]}
        lp = layout(8, k)
        res["layouts"][k] = {"lpcPitch": "uniform %d" % lp[0] if min(lp) == max(lp) else "spread 2..%d" % max(lp),
                             "ms_per_call_median": med, "ms_per_call_rounds": t, "spread_ms": float(max(t) - min(t)),
                             "delta_vs_%s_ms" % kinds[0]: med - base, "delta_vs_%s_pct" % kinds[0]: 100.0 * (med - base) / base,
                             "pitch_stage_ms_rounds": {p: [r[p] for r in stages[k]] for p in PITCH_STAGES},
                             "stage_ms_median": st}
    return res


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
    res = {"tool": "stream_pitch_orders_bench", "card": card_info(args.device)}
    res["leg1"] = leg(vp, ("a", "b", "u9"), args.steps, args.rounds, args.device, args.seconds)
    res["leg2"] = leg(vp, ("a'", "c", "u51"), args.steps, args.rounds, args.device, args.seconds, reserve=100)
    res["card_after"] = card_info(args.device)
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
