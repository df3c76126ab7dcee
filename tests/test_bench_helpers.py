"""bench.py's host-side arithmetic (no GPU): the host-link bound, the committed probe logs it falls back to, the
instruction-mix roofline read from the newest committed ncu capture, and the output sample of --dump-outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_link_bound_is_the_slowest_of_the_three_terms():
    link = {"h2d": 50.0, "d2h": 50.0, "duplex": 80.0}
    # twice as many bytes up as down (float I/O of the chain): the upload alone bounds the step
    assert bench.link_bound(link, 100e9, 50e9) == pytest.approx(2.0)
    # equal bytes: the shared total rate does
    assert bench.link_bound(link, 60e9, 60e9) == pytest.approx(1.5)
    # a slow download direction
    assert bench.link_bound({"h2d": 100.0, "d2h": 10.0, "duplex": 200.0}, 10e9, 20e9) == pytest.approx(2.0)


def test_committed_probe_logs_cover_1_2_4_8_gpus():
    for n in (1, 2, 4, 8):
        link = bench.link_ceiling(n)
        assert link is not None and all(link[k] > 10.0 for k in ("h2d", "d2h", "duplex")), n
        assert link["duplex"] <= link["h2d"] + link["d2h"] + 1e-9   # both directions together never beat the two alone
        assert os.path.exists(link["file"])
    assert bench.link_ceiling(3) is None
    # the 8-GPU finding the end-to-end section of DESIGN.md rests on: the host serves 8 GPUs less than twice what it serves one
    assert bench.link_ceiling(8)["duplex"] < 2.0 * bench.link_ceiling(1)["duplex"]


def test_instruction_mix_capture_feeds_the_roofline():
    for wl in ("chain48", "chain44", "voc44", "pitch44"):
        w = bench.mix_capture(wl)
        assert w is not None and w["passes_captured"] >= 1, wl
        tot = w["total"]
        assert tot["thread_inst_per_sample"] > tot["fp64_ops_per_sample"] + tot["fp32_ops_per_sample"] > 0
        assert abs(sum(s["fp64_ops_per_sample"] for s in w["stages"].values()) - tot["fp64_ops_per_sample"]) < 1e-6
    peaks = {"fp64_fma_per_s": 18.3e12, "fp32_fma_per_s": 36.0e12}
    samples = 2048 * 60 * 48000
    m = bench.mix_roofline("chain48", samples, 500.0, peaks, 1965.0)
    assert m is not None and 0.3 < m["frac"] < 1.0 and m["lower_bound_ms"] == pytest.approx(m["frac"] * 500.0)
    # the FP64 term dominates the chain; a step as fast as the bound would read frac = 1
    assert bench.mix_roofline("chain48", samples, m["lower_bound_ms"], peaks, 1965.0)["frac"] == pytest.approx(1.0)
    assert bench.mix_roofline("no-such-workload", samples, 500.0, peaks, 1965.0) is None


def test_dump_sample_is_seeded_bounded_and_exact():
    S, n = 40, 3000
    out = np.arange(S * n, dtype=np.float32).reshape(S, n)
    budget = 4 * 2 * (2 * n)   # room for two whole rows per array
    a, what = bench.dump_sample(lambda s: out[s].copy(), S, n, budget=budget)
    b, _ = bench.dump_sample(lambda s: out[s].copy(), S, n, budget=budget)
    assert all(np.array_equal(a[k], b[k]) for k in a)          # same arguments, same sample
    assert sum(x.nbytes for x in a.values()) <= budget
    assert a["rows"].shape == (2, n) and what["row_offset"] == 0
    assert np.array_equal(a["rows"], out[what["streams"]])
    assert a["cols"].shape == (S, what["cols"]) and what["cols"] == 2 * n // S
    assert np.all(np.isin(a["cols"][0], out[0])) and np.all(np.diff(a["cols"][0]) > 0)
    # a stream larger than half the budget: a seeded window of one stream
    a, what = bench.dump_sample(lambda s: out[s].copy(), S, n, budget=4 * 2 * 1000)
    off = what["row_offset"]
    assert a["rows"].shape == (1, 1000) and np.array_equal(a["rows"][0], out[what["streams"][0], off:off + 1000])
    assert sum(x.nbytes for x in a.values()) <= 4 * 2 * 1000


@pytest.mark.gpu
def test_dump_outputs_are_what_the_timed_steps_returned(vp, tmp_path):
    """bench.py --dump-outputs at the smoke-size workload: two runs write the same sample, and it is the sample of what the
    engine returns for the same seeded inputs through the host-buffer call."""
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--steps", "2", "--warmup", "1", "--no-e2e",
           "--no-cpu", "--no-parity", "--no-stream"]
    got = []
    for d in ("a", "b"):
        res = subprocess.run(cmd + ["--dump-outputs", str(tmp_path / d)], capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-3000:]
        line = json.loads(res.stdout.strip().splitlines()[-1])
        assert line["steps"] == 2 and line["dump_outputs"]["dir"] == str(tmp_path / d)
        got.append({k: np.load(tmp_path / d / ("outL_%s.npy" % k)) for k in ("rows", "cols")})
    assert all(np.array_equal(got[0][k], got[1][k]) for k in got[0])
    wl = bench.WORKLOADS["tiny"]
    fs, B, S = wl["fs"], wl["B"], wl["streams"]
    n = int(fs * wl["seconds"]) // B * B
    voice, sl, _ = vp.synth_host(fs, S, n, flavour=0, first_stream=0, want_right=False)
    eng = vp.Engine(fs, B, S, n // B, params=vp.default_params())
    try:
        out, _ = eng.process(voice, sl, None, want_right=False)
    finally:
        eng.close()
    want, _ = bench.dump_sample(lambda s: out[s], S, n)
    assert sum(a.nbytes for a in got[0].values()) <= bench.DUMP_BYTES
    assert all(np.array_equal(got[0][k], want[k]) for k in want)
