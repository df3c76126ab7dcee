#!/usr/bin/env python3
"""Cost and parity of per-stream state snapshots (vp_engine_save_streams / vp_engine_load_streams), in one run:

  device:    the default bench workload (chain48: 2048 streams x 60 s @ 48 kHz, block 1024, full chain, device-resident) is
             run once, then 64 and 2048 streams are saved and loaded back into other slots, alternating. Save: host clock
             around the call (it waits for the GPU and returns with the blob in host memory). Load: host clock around the
             call and a vp_engine_sync (the scatter has run). Effective bytes/s = blob bytes over that time.
  streaming: BASELINE config 5 (4096 streams, block 128 at 44.1 kHz, one CUDA graph per block phase) with 0, 1 and 64
             stream moves (save from some slots, load into others) before every block, alternating round by round. Per
             block the host clock from the move request to the return of vp_engine_stream_block; p50 / p99 against the
             2.90 ms block period, and the graph captures made while timed.
  parity:    16 streams x 60 s @ 48 kHz, each moved to another slot at the middle of the run, against the CPU reference on
             the stream's whole input: audio SNR / max error and pitch decisions.

The card's name, power limit and clocks are read in the same run.

    python tools/stream_snapshot_bench.py [--out FILE]

Prints one JSON line (and writes it to --out). Writes nothing else."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from stream_params_bench import card_info  # noqa: E402  (tools/ is this script's directory)


def spread(S, k, shift=0):
    return [int((s + shift) % S) for s in np.linspace(0, S - 1, k).round()] if k < S else list(range(S))


def device_leg(vp, rounds, dev):
    fs, B, S = 48000.0, 1024, 2048
    n = int(fs * 60.0) // B * B
    nb = n // B
    eng = vp.Engine(fs, B, S, nb, device=dev)
    bufs = [eng.device_alloc(S * n * 4) for _ in range(3)]
    dv, dl, do = bufs
    eng.synth_device(0, 0, S, n, n, dv, dl, None)
    res = {"workload": "chain48: %d streams x %.1f s @ 48 kHz, block 1024, device-resident, after one 60 s call" % (S, n / fs),
           "timer": "host clock (save: the call, which waits for the GPU; load: the call + vp_engine_sync)", "counts": {}}
    try:
        eng.process_device(nb, dv, dl, None, do, None, n, sync=True)
        for k in (64, 2048):
            src, dst = spread(S, k), spread(S, k, shift=1)
            blob = eng.save_streams(src)  # warm-up: staging buffers allocated
            eng.load_streams(dst, blob)
            eng.sync()
            ts, tl = [], []
            for _ in range(rounds):
                t0 = time.perf_counter()
                blob = eng.save_streams(src)
                ts.append(time.perf_counter() - t0)
                t0 = time.perf_counter()
                eng.load_streams(dst, blob)
                eng.sync()
                tl.append(time.perf_counter() - t0)
            mb = len(blob)
            res["counts"][str(k)] = {"blob_bytes": mb, "bytes_per_stream": (mb - vp.VP_SNAPSHOT_HEADER_BYTES) / k,
                                     "save_ms_median": float(np.median(ts)) * 1e3, "load_ms_median": float(np.median(tl)) * 1e3,
                                     "save_ms": [t * 1e3 for t in ts], "load_ms": [t * 1e3 for t in tl],
                                     "save_GBps": mb / float(np.median(ts)) / 1e9, "load_GBps": mb / float(np.median(tl)) / 1e9}
    finally:
        for p in bufs:
            eng.device_free(p)
        eng.close()
    return res


def streaming_leg(vp, blocks, rounds, dev):
    fs, Bs, S = 44100.0, 128, 4096
    pool = 64
    v, l, _ = vp.synth_host(fs, 256, pool * Bs, flavour=0, first_stream=0, want_right=False)
    V, L = np.tile(v, (S // 256, 1)), np.tile(l, (S // 256, 1))
    eng = vp.Engine(fs, Bs, S, 1, device=dev)
    counts = (0, 1, 64)
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
                src = spread(S, k, shift=b % 97)
                eng.load_streams(spread(S, k, shift=b % 97 + 1), eng.save_streams(src))
            eng.stream_block()
            t = time.perf_counter() - t0
            b += 1
            return t
        for _ in range(300):
            block(0)
        for k in counts[1:]:  # staging buffers of each size
            block(k)
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
           "timer": "host clock from the move request (save + load) to the return of vp_engine_stream_block",
           "graph_captures_while_timed": captures, "moves": {}}
    for k, t in lat.items():
        a = np.array(t) * 1e3
        res["moves"][str(k)] = {"p50_ms": float(np.percentile(a, 50)), "p99_ms": float(np.percentile(a, 99)),
                                "max_ms": float(a.max()), "p99_within_period": bool(np.percentile(a, 99) < period)}
    return res


def parity_leg(vp, dev):
    from common import MAXABS_MAX, SNR_MIN_DB, compare_decisions, maxabs, oracle_decisions, reference_runs, snr_db
    fs, B, P = 48000.0, 1024, 16
    n = int(fs * 60.0) // B * B
    nb = n // B
    half = nb // 2
    v, l, _ = vp.synth_host(fs, P, n, flavour=0, first_stream=100, want_right=False)
    V, L = np.zeros((2 * P, n), np.float32), np.zeros((2 * P, n), np.float32)
    V[:P], L[:P] = v, l
    V[P:, half * B:], L[P:, half * B:] = v[:, half * B:], l[:, half * B:]
    ow, ol, _ = vp.synth_host(fs, P, half * B, flavour=2, first_stream=300, want_right=False)
    V[P:, :half * B], L[P:, :half * B] = ow, ol  # the slots' old users
    eng = vp.Engine(fs, B, 2 * P, nb - half, device=dev)
    items = [dict(keyPitch=s % 13, gainVoc=-2.0 * (s % 4), gainPitch=1.0 - s % 3, gainVoice=-60.0, gainSynth=-60.0) for s in range(P)]
    try:
        eng.set_stream_params(0, items + items)
        o1, _ = eng.process(V[:, :half * B], L[:, :half * B], want_right=False)
        f1 = [eng.pitch_frames(s) for s in range(P)]
        eng.load_streams(list(range(P, 2 * P)), eng.save_streams(list(range(P))))
        o2, _ = eng.process(V[:, half * B:], L[:, half * B:], want_right=False)
        f2 = [eng.pitch_frames(s) for s in range(P, 2 * P)]
    finally:
        eng.close()
    refs, kind = reference_runs([(fs, B, v[s], l[s], None, items[s]) for s in range(P)])
    worst_snr, worst_err, bad, frames = 1e9, 0.0, 0, 0
    for s in range(P):
        got = np.concatenate([o1[s], o2[P + s]])
        worst_snr = min(worst_snr, snr_db(refs[s]["outL"], got))
        worst_err = max(worst_err, maxabs(refs[s]["outL"], got))
        dec = compare_decisions(vp, oracle_decisions(refs[s]["pitch"]), f1[s] + f2[s])
        bad += dec.bad
        frames += dec.n
    return {"streams": P, "seconds": n / fs, "moved_at_block": half, "reference": kind, "worst_snr_db": worst_snr,
            "worst_max_abs_err": worst_err, "pitch_frames": frames, "decision_mismatches": bad,
            "ok": bool(worst_snr >= SNR_MIN_DB and worst_err <= MAXABS_MAX and bad == 0)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--stream-blocks", type=int, default=500, help="timed blocks per configuration and round")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import vocoderproject_b200 as vp
    res = {"tool": "stream_snapshot_bench", "card": card_info(args.device)}
    res["device"] = device_leg(vp, args.rounds, args.device)
    res["streaming"] = streaming_leg(vp, args.stream_blocks, 2, args.device)
    res["parity"] = parity_leg(vp, args.device)
    res["card_after"] = card_info(args.device)
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
