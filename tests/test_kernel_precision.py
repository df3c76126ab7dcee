"""Precision of the kernels, path by path, against a float64 restatement of what they compute.

The rest of the suite holds the engine's audio to the acceptance bar (SNR >= 80 dB, common.SNR_MIN_DB). The kernels deliver
far more, and a kernel that lost 50 dB would still pass there. This file closes that gap:

  1. `voc_reference` restates one vocoder frame in numpy float64 (LPC.cpp:44-148, VocoderProcess.cpp:116-124,193-276): the
     analysis window of each window type, the autocorrelation, the Levinson recursion, the residual energies EeVoice /
     EeSynth by the direct FIR sum, the gain over the last 10 processed frames, and the silence gate that skips a frame.
     On the CPU it must reproduce the C oracle's per-frame log; then it is trusted for the GPU checks.
  2. Every live vocoder frame of the engine (voc_frames) is held to a per-frame bound derived from the reference's own
     reflection coefficients, at every order boundary of the tuned / generic kernels, and the kernels that ran are named
     (CUDA kernel records of torch.profiler).
  3. The audio of each path is held to a floor measured on the B200 (measured worst minus 6 dB), pitch decisions bit-exact.
  4. The sample-rate edges: 88.2 / 96 / 176.4 / 192 kHz, and a rate above 192 kHz refused at prepare.
"""
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import refbind
from common import SNR_MIN_DB, assert_decisions, compare_decisions, oracle_decisions, reference_runs, snr_db

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = 2.0 ** -52
PI_VOC = 3.14159265  # VocoderProcess.cpp:13 (truncated pi of the "sine" window)

# the order boundaries of the kernels (vp_voc.cu): rows are at least 40 / 5 wide, so <= 40 / <= 5 rides the tuned kernels
# zero padded; 41 / 6 and above take k_voc_levinson and k_voc_synth_generic; a row above 40 / 13 or a frame above 88.2 kHz
# takes k_voc_autocorr. The plug-in's ranges are [2, 100] / [2, 30] (include/vp_engine.h).
ORDER_CASES = [(2, 5), (39, 5), (40, 5), (41, 5), (64, 5), (100, 5), (40, 2), (40, 6), (40, 12), (40, 30)]

# SAFETY of the per-frame bound (see test_voc_frames_at_order_boundaries). The largest ratio error / ((p + sqrt(wlen))
# 2^-52 cond) seen: numpy reference against the C oracle (CPU, every case of test_reference_reproduces_the_oracle_log) 3.2,
# at p = 2 on the rectangular "hann" analysis window; engine against the reference (NVIDIA B200, 1000 W power limit, every
# case of test_voc_frames_at_order_boundaries) 3.8. SAFETY = 16 leaves a factor of 4.
SAFETY = 16.0


# ---------------------------------------------------------------------------------------------------- float64 reference
def voc_windows(wlen, hop, hann):
    """(analysis, synthesis) window, VocoderProcess.cpp:95-135: "sine" = the same sine window twice, "hann" = no analysis
    window and the juce Hann table for synthesis; both scaled by 1/sqrt(2) at the 75 % overlap."""
    i = np.arange(wlen, dtype=np.float64)
    factor = 1.0 / np.sqrt(2.0) if abs((wlen - hop) / wlen - 0.75) < 1e-10 else 1.0
    if hann:
        return np.ones(wlen), (0.5 - 0.5 * np.cos(2.0 * i * np.pi / (wlen - 1))) * factor
    w = factor * np.sin((i + 0.5) * PI_VOC / wlen)
    return w, w


def levinson(r, order):
    """LPC.cpp:107-148 for every row of r [F][>= order + 1] at once: (a [F][order + 1] with a0 = 1 and the reference's sign,
    reflection coefficients k [F][order])."""
    F = r.shape[0]
    a = np.zeros((F, order + 1))
    k = np.zeros((F, order))
    small = np.abs(r[:, 0]) < 1e-9
    r0 = np.where(small, 1.0, r[:, 0])
    a[:, 0] = 1.0
    a[:, 1] = r[:, 1] / r0
    k[:, 0] = a[:, 1]
    for p in range(2, order + 1):
        ap = a[:, 1:p].copy()
        rho = np.sum(r[:, p - 1:0:-1] * ap, axis=1)
        ra = np.sum(r[:, 1:p] * ap, axis=1)
        kp = (r[:, p] - rho) / (r0 - ra)
        a[:, 1:p] = ap - kp[:, None] * ap[:, ::-1]
        a[:, p] = kp
        k[:, p - 1] = kp
    a[:, 1:] *= -1.0
    a[small] = 0.0
    a[small, 0] = 1.0
    k[small] = 0.0
    return a, k


def frame_lpc(X, order):
    """Autocorrelation (LPC.cpp:44-97, biased: / wlen), Levinson and residual energy of the windowed frames X [F][wlen]:
    (E [F], condition estimate prod 1 / (1 - k_i^2) [F]). E is the reference's direct sum over the zero-state FIR residual
    (VocoderProcess.cpp:235-251), not the kernels' closed form."""
    F, wlen = X.shape
    r = np.empty((F, order + 1))
    for m in range(order + 1):
        r[:, m] = np.sum(X[:, :wlen - m] * X[:, m:], axis=1) / wlen
    a, k = levinson(r, order)
    e = X.copy()
    for j in range(1, order + 1):
        e[:, j:] += a[:, j:j + 1] * X[:, :wlen - j]
    cond = np.prod(1.0 / (1.0 - k * k), axis=1)
    return np.sum(e * e, axis=1), cond


def ring_gated(x, sizes, B, nBlocks):
    """Per host block: the ring RMS of MyBuffer.cpp:258-261 below -60 dB (juce gainToDecibels, -100 dB floor)."""
    inSize = sizes["inSize"]
    c = np.concatenate([[0.0], np.cumsum(np.asarray(x, np.float64) ** 2)])
    out = np.zeros(nBlocks, bool)
    for b in range(nBlocks):
        hi = (b + 1) * B
        ssum = c[hi] - c[max(0, hi - inSize)]
        rms = np.sqrt(max(ssum, 0.0) / inSize)
        db = max(20.0 * np.log10(rms), -100.0) if rms > 0 else -100.0
        out[b] = db < -60.0
    return out


def voc_reference(fs, B, voice, synth, lpcVoice, lpcSynth, hann, sizes):
    """Every vocoder frame of one stream (vocBool on throughout): dict of gated [F], EeVoice, EeSynth, g and the per-frame
    relative bounds bV, bS, bG of test_voc_frames_at_order_boundaries (bound only; the values are the reference's)."""
    hop, wlen, lat = sizes["hopV"], sizes["wlenV"], sizes["latency"]
    n = len(voice) // B * B
    nBlocks = n // B
    F = (n + hop - 1) // hop
    u0 = np.arange(F) * hop
    blk = u0 // B
    gate = ring_gated(voice[:n], sizes, B, nBlocks) | ring_gated(synth[:n], sizes, B, nBlocks)
    gated = gate[blk]
    wA, _ = voc_windows(wlen, hop, hann)
    idx = u0[:, None] + np.arange(wlen)[None, :]

    def frames(x):  # delayed timeline: input time = u - latency, zeros outside the input
        xp = np.concatenate([np.zeros(lat), np.asarray(x[:n], np.float64), np.zeros(wlen)])
        return xp[idx] * wA[None, :]
    live = ~gated
    EeV = np.zeros(F)
    EeS = np.zeros(F)
    cV = np.ones(F)
    cS = np.ones(F)
    EeV[live], cV[live] = frame_lpc(frames(voice)[live], lpcVoice)
    EeS[live], cS[live] = frame_lpc(frames(synth)[live], lpcSynth)
    bV = SAFETY * (lpcVoice + np.sqrt(wlen)) * EPS * cV
    bS = SAFETY * (lpcSynth + np.sqrt(wlen)) * EPS * cS
    # gain (VocoderProcess.cpp:264-276, :301-327): histories of the last 10 processed frames, zero before the first
    g = np.zeros(F)
    bG = np.zeros(F)
    HV, HS, hb = [0.0] * 10, [0.0] * 10, [0.0] * 10
    cur = 0.0
    for f in range(F):
        if live[f]:
            HV = [EeV[f]] + HV[:9]
            HS = [EeS[f]] + HS[:9]
            hb = [bV[f] + bS[f]] + hb[:9]
            cur = np.sqrt(sum(HV) / sum(HS)) if EeS[f] > 1e-4 else 0.0
        g[f] = cur
        bG[f] = 0.5 * max(hb) + 32 * EPS
    return dict(gated=gated, EeVoice=EeV, EeSynth=EeS, g=g, bV=bV, bS=bS, bG=bG)


def max_ratio(got, ref, live, bound):
    """max over live frames of |got - ref| / (|ref| bound): <= 1 passes."""
    err = np.abs(np.asarray(got, np.float64)[live] - ref[live]) / np.maximum(np.abs(ref[live]), 1e-300)
    return float(np.max(err / bound[live])) if live.any() else 0.0


def check_voc_frames(vf, ref, what):
    """EeVoice / EeSynth / g of every live frame within the per-frame bound, gate decisions equal. Returns the largest
    ratio error / bound of each quantity."""
    assert len(vf["gated"]) == len(ref["gated"]), "%s: %d frames, reference %d" % (what, len(vf["gated"]), len(ref["gated"]))
    assert np.array_equal(vf["gated"].astype(bool), ref["gated"]), what + ": gate decisions differ"
    live = ~ref["gated"]
    assert live.sum() >= 0.9 * len(live), what + ": most frames gated, nothing to compare"
    out = {}
    for k, b in (("EeVoice", "bV"), ("EeSynth", "bS"), ("g", "bG")):
        out[k] = max_ratio(vf[k], ref[k], live, ref[b])
        assert out[k] <= 1.0, "%s: %s off by %.3g x its bound" % (what, k, out[k])
    return out


# ----------------------------------------------------------------------------------------- CPU: reference vs the oracle
class _Log:
    """The oracle's per-frame vocoder log in the engine's voc_frames form."""
    def __init__(self, voc):
        self.vf = dict(gated=np.array([v.gated for v in voc], np.uint8), EeVoice=np.array([v.EeVoice for v in voc]),
                       EeSynth=np.array([v.EeSynth for v in voc]), g=np.array([v.g for v in voc]))


CPU_ORDERS = [(40, 5), (2, 2), (41, 6), (100, 30)]


@pytest.mark.parametrize("fs", [44100.0, 48000.0])
@pytest.mark.parametrize("hann", [False, True], ids=["sine", "hann"])
@pytest.mark.parametrize("flavour", [0, 1])
def test_reference_reproduces_the_oracle_log(vp, oracle, fs, hann, flavour):
    """The numpy restatement against the C oracle's per-frame vocoder log (two float64 computations of the same frames in
    different orders of summation): every live frame within the per-frame bound, the same gate decisions, at the order
    sets of the boundaries (default, smallest, first generic, largest)."""
    B = 1024
    n = int(fs * 1.0) // B * B
    voice, sl, _ = vp.synth_host(fs, 1, n, flavour=flavour, first_stream=7000 + flavour, want_right=False)
    sizes = oracle.sizes_for(fs, B)
    oracle.set_window(hann)
    try:
        for ov, os_ in CPU_ORDERS:
            r = oracle.run(fs, B, voice[0], sl[0], params=refbind.default_params(lpcVoice=ov, lpcSynth=os_, pitchBool=0), log=True)
            ref = voc_reference(fs, B, voice[0], sl[0], ov, os_, hann, sizes)
            check_voc_frames(_Log(r["voc"]).vf, ref, "fs %g %s orders %d / %d" % (fs, "hann" if hann else "sine", ov, os_))
    finally:
        oracle.set_window(False)


def test_reference_bound_bites_on_cpu(vp, oracle):
    """The per-frame bound is tight enough to see a one-rounding-in-FP32 Levinson: the same reference with the
    autocorrelation rounded to float32 (what an FP32 dot product in the recursion does to its inputs) fails it."""
    fs, B = 48000.0, 1024
    n = int(fs * 1.0) // B * B
    voice, sl, _ = vp.synth_host(fs, 1, n, flavour=1, first_stream=7001, want_right=False)
    sizes = oracle.sizes_for(fs, B)
    ref = voc_reference(fs, B, voice[0], sl[0], 40, 5, False, sizes)
    hop, wlen, lat = sizes["hopV"], sizes["wlenV"], sizes["latency"]
    live = ~ref["gated"]
    u0 = np.arange(len(live))[live] * hop
    xp = np.concatenate([np.zeros(lat), voice[0].astype(np.float64), np.zeros(wlen)])
    X = xp[u0[:, None] + np.arange(wlen)[None, :]] * voc_windows(wlen, hop, False)[0][None, :]
    r = np.stack([np.sum(X[:, :wlen - m] * X[:, m:], axis=1) / wlen for m in range(41)], axis=1)
    a, _ = levinson(r.astype(np.float32).astype(np.float64), 40)
    e = X.copy()
    for j in range(1, 41):
        e[:, j:] += a[:, j:j + 1] * X[:, :wlen - j]
    E, ok = ref["EeVoice"][live], ref["EeVoice"][live] > 0
    bad = np.abs(np.sum(e * e, axis=1)[ok] - E[ok]) / E[ok] / ref["bV"][live][ok]
    assert bad.max() > 1e3


# ------------------------------------------------------------------------------------------------ GPU: kernel records
def launched_kernels(fn):
    """Names of the CUDA kernels that ran inside fn() (CUPTI kernel records through torch.profiler: every kernel of the
    process, the engine's included), so a boundary case cannot silently test the other kernel."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
    names = set()
    for e in prof.events():
        m = re.search(r"\b(k_\w+)(<[^(]*>)?", e.name)
        if m:
            names.add(m.group(1) + (m.group(2) or "").replace(" ", ""))
    return res, names


def has(names, base):
    return any(n == base or n.startswith(base + "<") for n in names)


def expected_voc_kernels(fs, ordV, ordS, rowV, rowS):
    """The vocoder kernels vp_voc.cu dispatches for a call whose streams all run at ordV / ordS on rows rowV / rowS wide
    (vp_launch_voc_autocorr / _levinson / _synth): rows are at least 40 / 5, the autocorrelation and the synthesis go by
    the rows, the uniform Levinson by the orders themselves (k_voc_levinson_static is the <40, 5> solver)."""
    ac = "k_voc_autocorr2" if (rowV <= 40 and rowS <= 13 and fs <= 88200.0) else "k_voc_autocorr"
    lev = "k_voc_levinson_static" if (ordV, ordS, rowV, rowS) == (40, 5, 40, 5) else "k_voc_levinson"
    syn = "k_voc_synth_rows" if (rowV, rowS) == (40, 5) else "k_voc_synth_generic"
    return ac, lev, syn


def assert_voc_kernels(names, fs, ordV, ordS, rowV=None, rowS=None):
    rowV, rowS = rowV or max(ordV, 40), rowS or max(ordS, 5)
    want = expected_voc_kernels(fs, ordV, ordS, rowV, rowS)
    every = ("k_voc_autocorr2", "k_voc_autocorr", "k_voc_levinson_static", "k_voc_levinson", "k_voc_synth_rows",
             "k_voc_synth_generic")
    for k in every:
        assert has(names, k) == (k in want), "kernel %s %s at %g Hz, orders %d / %d on rows %d / %d (launched: %s)" % (
            k, "missing" if k in want else "ran", fs, ordV, ordS, rowV, rowS, sorted(names))


def engine_run(vp, fs, B, voice, sl, sr, params, **kw):
    S, n = voice.shape

    def go():
        eng = vp.Engine(fs, B, S, n // B, params=vp.default_params(**params), **kw)
        try:
            outL, outR = eng.process(voice, sl, sr)
            return outL, outR, [eng.voc_frames(s) for s in range(S)], [eng.pitch_frames(s) for s in range(S)], eng.sizes
        finally:
            eng.close()
    return launched_kernels(go)


# ---------------------------------------------------------------------------------- GPU: per-frame vocoder at the boundaries
@pytest.mark.gpu
@pytest.mark.parametrize("fs", [44100.0, 48000.0])
@pytest.mark.parametrize("hann", [False, True], ids=["sine", "hann"])
@pytest.mark.parametrize("orders", ORDER_CASES, ids=["%d-%d" % o for o in ORDER_CASES])
def test_voc_frames_at_order_boundaries(vp, fs, hann, orders):
    """EeVoice, EeSynth and g of every live frame against the float64 reference, on the voice with the -80 dBFS noise floor
    (flavour 1, the FP64 stress case) and the default one (flavour 0), 1.5 s each.

    The bound, per frame and quantity, relative: SAFETY x (p + sqrt(wlen)) x 2^-52 x prod_i 1 / (1 - k_i^2), k_i the
    reference's own reflection coefficients at the frame's order p. Why: the residual energy of order p is
    E_p = r0 prod (1 - k_i^2), so the product is r0 / E_p, the prediction gain. Every rounding the kernel and the reference
    make differently is a relative error of a few 2^-52 on a quantity of size r0, i.e. of up to that many r0 2^-52 on E_p,
    which relative to E_p is multiplied by r0 / E_p. The recursion makes one such rounding per order (p); the
    autocorrelation lags and the residual energy are sums of wlen terms, whose roundings in different orders of summation
    (segments and FMA chains on the GPU, pairwise in numpy, the kernels' closed form E = wlen (r0 + sum a_k r_k) - tail
    against the direct FIR sum) differ like a random walk, sqrt(wlen) units. The order alone is not enough: at p = 2 on
    the rectangular analysis window of "hann" the two float64 computations differ by 40 p 2^-52 r0 / E_p. SAFETY = 16 is
    above what both pairs of float64 computations were measured to need (the constant's comment). The gain
    g = sqrt(sum of 10 EeVoice / sum of 10 EeSynth) of positive terms inherits half the sum of the worst EeVoice and
    EeSynth bounds over its 10 frames, plus the roundings of its sums and square root (32 x 2^-52). A kernel that drops a
    lag or rounds one dot product to FP32 misses this by orders of magnitude (test_reference_bound_bites_on_cpu; the
    mutation table of DESIGN section 6)."""
    ov, os_ = orders
    B = 1024
    n = int(fs * 1.5) // B * B
    v0, l0, r0 = vp.synth_host(fs, 1, n, flavour=0, first_stream=7100 + ov)
    v1, l1, r1 = vp.synth_host(fs, 1, n, flavour=1, first_stream=7200 + os_)
    voice, sl, sr = np.concatenate([v0, v1]), np.concatenate([l0, l1]), np.concatenate([r0, r1])
    (_, _, vfs, _, sizes), names = engine_run(vp, fs, B, voice, sl, sr, dict(lpcVoice=ov, lpcSynth=os_, pitchBool=0),
                                              window=vp.VP_WINDOW_HANN if hann else vp.VP_WINDOW_SINE)
    assert_voc_kernels(names, fs, ov, os_)
    worst = {}
    for s in range(2):
        ref = voc_reference(fs, B, voice[s], sl[s], ov, os_, hann, sizes)
        got = check_voc_frames(vfs[s], ref, "stream %d (flavour %d)" % (s, s))
        for k, v in got.items():
            worst[k] = max(worst.get(k, 0.0), v)
    print("PRECISION voc fs=%g %s orders=%d/%d ratio EeV %.3g EeS %.3g g %.3g" % (
        fs, "hann" if hann else "sine", ov, os_, worst["EeVoice"], worst["EeSynth"], worst["g"]))


@pytest.mark.gpu
@pytest.mark.parametrize("fs", [44100.0, 48000.0])
def test_mixed_batch_on_generic_kernels(vp, fs):
    """Streams at 40 / 5 beside one at 41 / 6: the call's rows are 41 / 6 wide, so the 40 / 5 streams run the generic
    autocorrelation, Levinson and synthesis on zero-padded rows. Each stream against the reference at its own orders."""
    B, S = 1024, 3
    n = int(fs * 1.5) // B * B
    voice, sl, sr = vp.synth_host(fs, S, n, flavour=1, first_stream=7300)
    orders = [(40, 5), (40, 5), (41, 6)]

    def go():
        eng = vp.Engine(fs, B, S, n // B, params=vp.default_params(pitchBool=0), reserve_orders=(41, 6))
        try:
            eng.set_stream_orders(0, orders)
            eng.process(voice, sl, sr)
            return [eng.voc_frames(s) for s in range(S)], eng.sizes
        finally:
            eng.close()
    (vfs, sizes), names = launched_kernels(go)
    assert_voc_kernels(names, fs, 40, 5, 41, 6)  # (the 40 / 5 streams: generic on 41 / 6 rows)
    for s, (ov, os_) in enumerate(orders):
        check_voc_frames(vfs[s], voc_reference(fs, B, voice[s], sl[s], ov, os_, False, sizes), "stream %d at %d / %d" % (s, ov, os_))


# ------------------------------------------------------------------------------------------------ GPU: audio floors
# Worst stream's SNR against the reference (reference_runs: the reference's strict build where present, else the C port
# that is bit-identical to it), per path, over the streams of FLOOR_CASES. Floor = measured worst - 6 dB. Measured on an
# NVIDIA B200 at a 1000 W power limit (the figure in each comment); every path but rows32 sits at the ~146 dB that rounding
# the output to float32 leaves, so a path that loses more than 6 dB of its FP64 precision fails here.
FLOORS = {
    "tuned44": 139.6,      # 145.67 dB
    "tuned48": 139.4,      # 145.46 dB
    "orders24_8": 139.6,   # 145.65 dB
    "orders20_3": 139.7,   # 145.79 dB
    "orders64_12": 139.6,  # 145.65 dB
    "pitch2": 139.6,       # 145.66 dB
    "pitch16": 139.7,      # 145.77 dB
    "pitch100": 139.5,     # 145.57 dB
    "rows32": 122.9,       # 128.94 dB (VP_SYNTH=rows32: FP32 whitening FIR and window multiplies)
    "fs96": 139.6,         # 145.69 dB
    "fs176": 139.8,        # 145.87 dB
    "fs192": 139.7,        # 145.71 dB
}

FLOOR_CASES = {
    # name: (fs, streams, seconds, flavours, params, synth variant)
    "tuned44": (44100.0, 3, 2.0, (0, 1, 0), dict(keyPitch=3), "rows"),
    "tuned48": (48000.0, 3, 2.0, (0, 1, 0), dict(), "rows"),
    "orders24_8": (44100.0, 3, 2.0, (0, 1, 0), dict(lpcVoice=24, lpcSynth=8, lpcPitch=20), "rows"),
    "orders20_3": (44100.0, 3, 2.0, (0, 1, 0), dict(lpcVoice=20, lpcSynth=3, lpcPitch=9), "rows"),
    "orders64_12": (44100.0, 3, 2.0, (0, 1, 0), dict(lpcVoice=64, lpcSynth=12, lpcPitch=30), "rows"),
    "pitch2": (44100.0, 3, 2.0, (0, 0, 0), dict(lpcPitch=2, keyPitch=3), "rows"),
    "pitch16": (44100.0, 3, 2.0, (0, 0, 0), dict(lpcPitch=16), "rows"),
    "pitch100": (44100.0, 3, 2.0, (0, 0, 0), dict(lpcPitch=100, keyPitch=7), "rows"),
    "rows32": (48000.0, 3, 2.0, (0, 1, 0), dict(), "rows32"),
    "fs96": (96000.0, 1, 1.2, (0,), dict(keyPitch=3), "rows"),
    "fs176": (176400.0, 1, 1.0, (0,), dict(), "rows"),
    "fs192": (192000.0, 1, 1.0, (0,), dict(keyPitch=5), "rows"),
}

_CHILD = r"""
import sys, numpy as np
sys.path[:0] = [%r]
import vocoderproject_b200 as vp
d = np.load(sys.argv[1])
eng = vp.Engine(float(d["fs"]), int(d["B"]), d["voice"].shape[0], d["voice"].shape[1] // int(d["B"]),
                params=vp.default_params(**{k: int(v) for k, v in zip(d["pk"], d["pv"])}))
outL, outR = eng.process(d["voice"], d["sl"], d["sr"])
np.save(sys.argv[2], outL)
eng.close()
"""


def floor_inputs(vp, fs, S, secs, flavours, B, first):
    n = int(fs * secs) // B * B
    parts = [vp.synth_host(fs, 1, n, flavour=f, first_stream=first + i) for i, f in enumerate(flavours[:S])]
    return tuple(np.concatenate([p[j] for p in parts]) for j in range(3))


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(FLOOR_CASES))
def test_audio_floor_per_path(vp, name):
    """Worst stream's SNR of each path against the reference at the floor that path was measured to deliver, and every
    pitch decision bit-exact (outside flagged frames, as everywhere in the suite)."""
    fs, S, secs, flavours, params, synth = FLOOR_CASES[name]
    B = 1024
    voice, sl, sr = floor_inputs(vp, fs, S, secs, flavours, B, 7400 + 10 * sorted(FLOOR_CASES).index(name))
    if synth == "rows32":
        # VP_SYNTH is read once per process (vp_voc.cu: vs_variant): the rows32 build of the synthesis runs in a child
        with tempfile.TemporaryDirectory() as td:
            inp, outp = os.path.join(td, "in.npz"), os.path.join(td, "out.npy")
            np.savez(inp, fs=fs, B=B, voice=voice, sl=sl, sr=sr, pk=list(params), pv=[int(v) for v in params.values()])
            env = dict(os.environ, VP_SYNTH="rows32")
            subprocess.check_call([sys.executable] + (["-s"] if sys.flags.no_user_site else []) +
                                  ["-c", _CHILD % ROOT, inp, outp], env=env, cwd=ROOT)
            outL, pfs = np.load(outp), None
    else:
        (outL, _, _, pfs, _), names = engine_run(vp, fs, B, voice, sl, sr, params)
        if fs > 48000.0:  # tauMax > 480: the shared-memory YIN decision instead of the register-resident one
            assert has(names, "k_yin_decide") and not has(names, "k_yin_decide_reg"), sorted(names)
        if params.get("lpcPitch", 15) != 15:
            for k in ("k_pitch_levinson", "k_pitch_psola", "k_pitch_iir"):
                assert any(n.startswith(k + "<0") for n in names) and not any(n.startswith(k + "<15") for n in names), (k, sorted(names))
    refs, kind = reference_runs([(fs, B, voice[s], sl[s], sr[s], params) for s in range(S)])
    snrs = [snr_db(r["outL"], outL[s]) for s, r in enumerate(refs)]
    worst, floor = min(snrs), FLOORS[name]
    print("PRECISION floor %s worst %.2f dB (streams %s) against %s" % (name, worst, ["%.2f" % x for x in snrs], kind))
    assert worst >= floor, "%s: worst stream %.1f dB, floor %.1f dB" % (name, worst, floor)
    if pfs is not None:
        for s, r in enumerate(refs):
            assert r.get("ub", 0) == 0
            assert_decisions(compare_decisions(vp, oracle_decisions(r["pitch"]), pfs[s]), "%s stream %d" % (name, s))


# ----------------------------------------------------------------------------------------------- GPU: sample-rate edges
@pytest.mark.gpu
@pytest.mark.parametrize("fs", [88200.0, 96000.0])
def test_either_side_of_the_autocorrelation_switch(vp, oracle, fs):
    """88.2 kHz is the highest of the common rates whose vocoder frames fit the tuned autocorrelation's shared memory, 96 kHz
    the lowest that takes k_voc_autocorr; above 48 kHz (tauMax > 480) the YIN decision is the shared-memory k_yin_decide on
    both. Audio and every pitch decision against the oracle, per-frame vocoder values against the float64 reference."""
    B = 1024
    n = int(fs * 1.0) // B * B
    voice, sl, sr = vp.synth_host(fs, 1, n, flavour=0, first_stream=7500)
    (outL, _, vfs, pfs, sizes), names = engine_run(vp, fs, B, voice, sl, sr, dict(keyPitch=3))
    assert_voc_kernels(names, fs, 40, 5)
    assert has(names, "k_yin_decide") and not has(names, "k_yin_decide_reg"), sorted(names)
    r = oracle.run(fs, B, voice[0], sl[0], synthR=sr[0], params=refbind.default_params(keyPitch=3), log=True)
    assert r["ub"] == 0
    assert snr_db(r["outL"], outL[0]) >= (FLOORS["fs96"] if fs == 96000.0 else SNR_MIN_DB)  # 88.2 kHz: not measured
    assert_decisions(compare_decisions(vp, oracle_decisions(r["pitch"]), pfs[0]), "fs %g" % fs)
    check_voc_frames(vfs[0], voc_reference(fs, B, voice[0], sl[0], 40, 5, False, sizes), "fs %g" % fs)


@pytest.mark.gpu
def test_rate_above_192k_is_refused_at_prepare(vp):
    """192 kHz is the top of the supported range (tauMax <= 1920, vp_engine_prepare); just above it prepare answers
    VP_E_ARG before it allocates anything: the engine stays unprepared (its layout query answers VP_E_STATE)."""
    import ctypes as C
    assert vp.sizes_for(192000.0, 1024)["tauMax"] == 1920
    lib = vp.load_library()
    h = C.c_void_p()
    assert lib.vp_engine_create(C.byref(h), 0) == vp.VP_OK
    try:
        p = vp.default_params()
        assert lib.vp_engine_set_params(h, C.byref(p)) == vp.VP_OK
        assert lib.vp_engine_prepare(h, 192001.0, 1024, 1, 8, 0) == vp.VP_E_ARG
        a, b, c = C.c_int(0), C.c_int(0), C.c_size_t(0)
        assert lib.vp_engine_get_info(h, C.byref(a), C.byref(b), C.byref(c)) == vp.VP_E_STATE
        assert c.value == 0
        # the same engine then prepares at 192 kHz
        assert lib.vp_engine_prepare(h, 192000.0, 1024, 1, 8, 0) == vp.VP_OK
        assert lib.vp_engine_get_info(h, C.byref(a), C.byref(b), C.byref(c)) == vp.VP_OK and c.value > 0
    finally:
        lib.vp_engine_destroy(h)
