#!/usr/bin/env python3
"""Cost of per-stream resets (vp_engine_reset_streams), three measurements in one run:

  device:    the default bench workload (chain48: 2048 streams x 60 s @ 48 kHz, block 1024, full chain, device-resident) with
             0, 64 and 2048 streams reset before each call, alternating round by round. Step = vp_engine_reset, the stream
             resets, one process call over the whole batch, timed with CUDA events on the engine's stream.
  streaming: BASELINE config 5 (4096 streams, block 128 at 44.1 kHz, one CUDA graph per block phase) with 0, 1, 64 and 4096
             streams reset before every block, alternating round by round. Per block the host clock from the reset request
             to the return of vp_engine_stream_block (which waits for the block's output); p50 / p99 against the 2.90 ms
             block period.
  kernel:    k_reset_streams alone, from the CUDA activity trace of torch.profiler in a section of its own (64, 2048 and
             4096 streams listed): the engine launches it on its own stream, where no event of the caller's can bracket it.

The card's name, power limit and clocks are read in the same run.

    python tools/reset_streams_bench.py [--out FILE]

Prints one JSON line (and writes it to --out). Writes nothing else."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from stream_params_bench import card_info  # noqa: E402  (tools/ is this script's directory)


def spread(S, k):
    return [int(s) for s in np.linspace(0, S - 1, k).round()] if k < S else list(range(S))


def device_leg(vp, steps, rounds, dev):
    fs, B, S = 48000.0, 1024, 2048
    n = int(fs * 60.0) // B * B
    nb = n // B
    eng = vp.Engine(fs, B, S, nb, device=dev)
    bufs = [eng.device_alloc(S * n * 4) for _ in range(3)]
    dv, dl, do = bufs
    eng.synth_device(0, 0, S, n, n, dv, dl, None)
    counts = (0, 64, 2048)
    times = {k: [] for k in counts}

    def step(k):
        eng.reset()
        if k:
            eng.reset_streams(spread(S, k))
        eng.process_device(nb, dv, dl, None, do, None, n, sync=False)
    try:
        for _ in range(rounds):
            for k in counts:
                step(k)  # warm-up step of this configuration
                eng.sync()
                eng.timer_record(0)
                for _ in range(steps):
                    step(k)
                eng.timer_record(1)
                eng.sync()
                times[k].append(eng.timer_elapsed_ms(0, 1) / steps)
        sp = eng.info()["streams_per_pass"]
    finally:
        for p in bufs:
            eng.device_free(p)
        eng.close()
    res = {"workload": "chain48: %d streams x %.1f s @ 48 kHz, block 1024, device-resident" % (S, n / fs), "streams_per_pass": sp,
           "steps_per_round": steps, "rounds": rounds,
           "timer": "CUDA events on the engine's stream around each round's steps (reset + stream resets + one process call)",
           "resets": {}}
    base = float(np.median(times[0]))
    for k, t in times.items():
        med = float(np.median(t))
        res["resets"][str(k)] = {"ms_per_step_median": med, "ms_per_step_rounds": t, "spread_ms": float(max(t) - min(t)),
                                 "delta_vs_0_ms": med - base}
    return res


def streaming_leg(vp, blocks, rounds, dev):
    fs, Bs, S = 44100.0, 128, 4096
    pool = 64  # blocks of distinct input, cycled
    v, l, _ = vp.synth_host(fs, 256, pool * Bs, flavour=0, first_stream=0, want_right=False)
    V, L = np.tile(v, (S // 256, 1)), np.tile(l, (S // 256, 1))
    eng = vp.Engine(fs, Bs, S, 1, device=dev)
    counts = (0, 1, 64, 4096)
    lat = {k: [] for k in counts}
    try:
        hv, hs, _ = eng.stream_buffers()
        b = 0

        def block(k, lists):
            nonlocal b
            x = slice((b % pool) * Bs, (b % pool + 1) * Bs)
            hv[:] = V[:, x]
            hs[:] = L[:, x]
            t0 = time.perf_counter()
            if k:
                eng.reset_streams(lists[b % len(lists)])
            eng.stream_block()
            t = time.perf_counter() - t0
            b += 1
            return t
        lists = {k: [spread(S, k)] if k != 1 else [[s] for s in range(0, S, 97)] for k in counts}
        for _ in range(300):  # every block phase captured, clocks up
            block(0, None)
        cap0 = eng.stream_stats()["graph_captures"]
        for _ in range(rounds):
            for k in counts:
                for _ in range(blocks):
                    lat[k].append(block(k, lists.get(k)))
        captures_after_warmup = eng.stream_stats()["graph_captures"] - cap0
    finally:
        eng.close()
    period = Bs / fs * 1e3
    res = {"workload": "BASELINE config 5: %d streams, block %d @ 44.1 kHz, CUDA graph per block phase" % (S, Bs),
           "block_period_ms": period, "blocks_per_config": blocks * rounds, "rounds": rounds,
           "timer": "host clock from the reset request to the return of vp_engine_stream_block (the block's output is in host memory)",
           "graph_captures_while_timed": captures_after_warmup, "resets": {}}
    for k, t in lat.items():
        a = np.array(t) * 1e3
        res["resets"][str(k)] = {"p50_ms": float(np.percentile(a, 50)), "p99_ms": float(np.percentile(a, 99)),
                                 "max_ms": float(a.max()), "p99_within_period": bool(np.percentile(a, 99) < period)}
    return res


def kernel_leg(vp, dev):
    """k_reset_streams' device time in the profiler's CUDA activity trace, per listed-stream count."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    out = {}
    for fs, B, S, ks in ((48000.0, 1024, 2048, (64, 2048)), (44100.0, 128, 4096, (64, 4096))):
        eng = vp.Engine(fs, B, S, 1, device=dev)
        try:
            hv, hs, _ = eng.stream_buffers()
            for _ in range(30):
                eng.stream_block()
            for k in ks:
                eng.reset_streams(spread(S, k))  # warm-up launch of this size
                eng.stream_block()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(20):
                        eng.reset_streams(spread(S, k))
                        eng.stream_block()
                us = [e.device_time_total / e.count for e in prof.key_averages() if "k_reset_streams" in e.key]
                h = eng.info()["history_samples"]
                out["%g Hz B=%d: %d of %d streams" % (fs, B, k, S)] = {
                    "kernel_us": us[0] if us else None, "launches": 20, "history_samples": h}
        finally:
            eng.close()
    return {"timer": "torch.profiler CUDA activity trace (CUPTI kernel records), mean over 20 launches", "configs": out}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--stream-blocks", type=int, default=500, help="timed blocks per configuration and round")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import vocoderproject_b200 as vp
    res = {"tool": "reset_streams_bench", "card": card_info(args.device)}
    res["device"] = device_leg(vp, args.steps, args.rounds, args.device)
    res["streaming"] = streaming_leg(vp, args.stream_blocks, args.rounds, args.device)
    res["kernel"] = kernel_leg(vp, args.device)
    res["card_after"] = card_info(args.device)
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
