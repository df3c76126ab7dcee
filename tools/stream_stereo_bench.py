#!/usr/bin/env python3
"""Latency of stereo streaming (vp_engine_stream_buffers_stereo) against mono streaming, in one run.

Workload: the streaming sub-test of bench.py (BASELINE config 5): 4096 streams, block 128 @ 44.1 kHz, default parameters,
64 pre-generated blocks cycled, graphs of every block phase captured over the first 32 blocks, then 1500 timed blocks
per layout and round. Four layouts, one engine each, all in this process, run alternately round by round:

  a_mono          the mono buffers (vp_engine_stream_buffers): voice + synthL in, outL out;
  b_stereo        the stereo buffers, no stream with the dry side-chain on;
  c_stereo_dry10  the stereo buffers, dry side-chain (gainSynth -12 dB) on every 10th stream;
  d_stereo_dry    the stereo buffers, dry side-chain on every stream.

Per layout: p50 / p99 / max of the host clock around vp_engine_stream_block (pinned H2D + graph + pinned D2H + sync), and
the graph captures (during the warm-up, with the slowest warm-up block, which includes a capture, and while timed).
Stereo adds 2 x 4096 x 128 x 4 B = 4 MiB of link traffic per block. The card's name, power limit and max SM clock are read in the same run (nvidia-smi --query-gpu, read-only).

    python tools/stream_stereo_bench.py [--rounds 3] [--blocks 1500] [--out FILE]

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

LAYOUTS = {"a_mono": (False, None), "b_stereo": (True, None), "c_stereo_dry10": (True, 10), "d_stereo_dry": (True, 1)}


class Leg:
    """One engine streaming one layout; block() feeds the next of the cycled input blocks and times stream_block."""

    def __init__(self, vp, fs, B, S, stereo, dry_every, src, dev):
        self.B, self.src, self.b = B, src, 0
        self.eng = vp.Engine(fs, B, S, 1, params=vp.default_params(), device=dev)
        if dry_every:
            self.eng.set_stream_params(0, [dict(gainSynth=-12.0 if s % dry_every == 0 else -60.0) for s in range(S)])
        bufs = self.eng.stream_buffers(stereo=stereo)
        self.hv, self.hs = bufs[0], bufs[1]
        self.hr = bufs[2] if stereo else None
        self.lat, self.warm = [], []

    def block(self, timed):
        V, L, R = self.src
        x = slice((self.b % 64) * self.B, (self.b % 64 + 1) * self.B)
        self.hv[:] = V[:, x]
        self.hs[:] = L[:, x]
        if self.hr is not None:
            self.hr[:] = R[:, x]
        t0 = time.perf_counter()
        self.eng.stream_block()
        t = time.perf_counter() - t0
        self.b += 1
        (self.lat if timed else self.warm).append(t * 1e3)

    def captures(self):
        return self.eng.stream_stats()["graph_captures"]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--blocks", type=int, default=1500, help="timed blocks per layout and round")
    ap.add_argument("--warm", type=int, default=32, help="untimed blocks per layout before the first round")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import vocoderproject_b200 as vp
    fs, B, S = 44100.0, 128, 4096
    res = {"tool": "stream_stereo_bench", "card": card_info(args.device)}
    v, l, r = vp.synth_host(fs, 64, 64 * B, flavour=0, first_stream=0)
    reps = S // 64
    src = tuple(np.tile(a, (reps, 1)) for a in (v, l, r))
    legs = {name: Leg(vp, fs, B, S, st, dry, src, args.device) for name, (st, dry) in LAYOUTS.items()}
    try:
        for leg in legs.values():
            for _ in range(args.warm):
                leg.block(False)
        warm_caps = {k: leg.captures() for k, leg in legs.items()}
        per_round = args.blocks
        for _ in range(args.rounds):
            for leg in legs.values():
                for _ in range(per_round):
                    leg.block(True)
        caps = {k: leg.captures() for k, leg in legs.items()}
    finally:
        for leg in legs.values():
            leg.eng.close()
    period = B / fs * 1e3
    res["workload"] = "BASELINE config 5: %d streams, block %d @ 44.1 kHz, default parameters, CUDA graph per block phase" % (S, B)
    res["timer"] = "host perf_counter around vp_engine_stream_block (pinned H2D + graph + pinned D2H + sync)"
    res["block_period_ms"] = period
    res["rounds"], res["blocks_per_layout"] = args.rounds, per_round * args.rounds
    res["extra_link_bytes_per_block_stereo"] = 2 * S * B * 4
    res["layouts"] = {}
    for k, leg in legs.items():
        a = np.array(leg.lat)
        res["layouts"][k] = {"p50_ms": float(np.percentile(a, 50)), "p99_ms": float(np.percentile(a, 99)), "max_ms": float(a.max()),
                             "mean_ms": float(a.mean()), "graph_captures_warmup": warm_caps[k],
                             "warmup_max_ms": float(max(leg.warm)),
                             "graph_captures_while_timed": caps[k] - warm_caps[k],
                             "p99_by_round_ms": [float(np.percentile(a[i * per_round:(i + 1) * per_round], 99)) for i in range(args.rounds)]}
    res["card_after"] = card_info(args.device)
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
