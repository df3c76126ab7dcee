"""YIN's period decision at the edges of its FP32 arithmetic.

The reference (PitchProcess.cpp:350-448, restated in oracle/vp_oracle.c: yin) sums (x[i] - x[i+k])^2 in double. The engine
computes d[k] = A + B(k) - 2 C(k) with C(k) accumulated in FP32 (k_yin_corr), checks every deciding comparison against a
bound on that accumulation's error (k_yin_decide_reg, k_yin_decide) and sends a frame whose comparisons are inside the
bound to the FP64 direct-form kernel (k_yin<R, double>). VP_YIN_MODE=direct uses the FP32 direct form (k_yin<R, float>)
with its own re-check criterion instead. Bit-exact pitch decisions rest on those bounds being rigorous; the inputs here
push them:
  ladder     stretches of a voice scaled by 2^-k, loud audio on both sides (FP32 underflow, k up to FP32 subnormals),
  dc         DC + a voice (cancellation in A + B - 2C; most frames must go to FP64),
  threshold  the CMND of the dip within 1e-1 .. 1e-6 (relative) of yinTol on either side,
  edges      periods T + 0.5 (d'(T) ~ d'(T + 1) in the descent) and exact periods at tauMin, tauMin + 1, the two-phase
             split (lag 240), tauMax - 2 and tauMax - 1 (U3: the descent reads yinTemp[tauMax]).
Every family runs as one batch through the C ABI and is compared with the oracle frame by frame, on the default two-phase
path, one pass over all lags (VP_YIN_PHASES=1) and the FP32 direct form (VP_YIN_MODE=direct), at 44.1 / 48 kHz (register
decision kernels, two phases) and 96 kHz (generic decision kernel). The CPU tests pin the restatement, the premises of the
inputs and the error bound itself."""
import math
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import oraclebind
import refbind
from common import MAXABS_MAX, SNR_MIN_DB, kat_inputs, maxabs, oracle_decisions, snr_db

YIN_TOL = 0.25
RATES = {"44k": (44100.0, 1024), "48k": (48000.0, 1024), "96k": (96000.0, 1024)}
LADDER = (0, 20, 40, 60, 64, 66, 68, 70, 72, 75, 80, 100, 120, 140)
DC_CASES = ((0.0, 1.0), (0.5, 0.05), (0.9, 0.01), (0.95, 0.002))
FAMILIES = ("ladder", "dc", "threshold", "edges")
PATHS = ("two_phase", "single_pass", "direct")
DC_STREAMS = 128      # per (DC, a) case: 512 streams, the heaviest case alone fills several rounds of the re-check grid
LADDER_MIN_FRAMES = 8  # ungated frames per stream that lie entirely inside a scaled stretch

# FP32 accumulation error of one C(k) (vocoderproject_b200/csrc/vp_pitch.cu: yin_corr_beta, yin_corr_abs): YC_SUB first-level
# terms, relative part beta(c) (A + B(k)) of |err d[k]|, and per rounding at most 2^-150 absolute in the subnormal range.
YC_SUB = 60


def corr_beta(c):
    return (YC_SUB + c // YC_SUB + 4) * 2.0 ** -24 * 1.25


def corr_abs(c):
    return 2.0 * 4 * (c + c // YC_SUB + 2) * 2.0 ** -150 * 1.25


# ---------------------------------------------------------------------------------------------------------------------
# geometry, restatement


def geom(fs, B):
    """The oracle's sizes plus tauMin (floor(fs / fMax), PitchProcess.cpp:429) and the YIN window length."""
    z = dict(oraclebind.sizes_for(fs, B))
    z["tauMin"] = int(math.floor(fs / 800.0))
    z["win"] = z["frameLenP"] + z["tauMax"] - 1
    z["fs"], z["B"] = fs, B
    return z


def frame_window(x, z, row):
    """The samples yin() reads for a logged frame: x[p - tauMax + i + k] on the delayed timeline, i < L, k < tauMax,
    i.e. input samples [p - latency - tauMax, + L + tauMax - 1); zero outside the input (the rings start zeroed)."""
    p = row.block * z["B"] + row.startSample
    w0 = p - z["latency"] - z["tauMax"]
    out = np.zeros(z["win"])
    a, b = max(w0, 0), min(w0 + z["win"], len(x))
    if b > a:
        out[a - w0:b - w0] = x[a:b]
    return out, w0


def yin64(w, z):
    """Float64 restatement of the oracle's yin() on one window: (period, margin, u3).
    margin = the smallest relative distance of any deciding comparison: |d' - tol| / tol for every lag from tauMin up to
    the first one under the threshold, |d'(k+1) - d'(k)| / |d'(k)| along the descent. u3: the descent starts at
    tauMax - 1 and reads yinTemp[tauMax] (SURVEY App. B U3)."""
    L, tauMin, tauMax = z["frameLenP"], z["tauMin"], z["tauMax"]
    x = np.asarray(w, np.float64)
    lagged = np.lib.stride_tricks.sliding_window_view(x, L)[:tauMax]  # row k = x[k : k + L]
    d = ((x[:L] - lagged) ** 2).sum(axis=1)
    k = np.arange(tauMax, dtype=np.float64)
    run = np.cumsum(d[1:])
    dn = np.ones(tauMax)
    with np.errstate(invalid="ignore", divide="ignore"):
        dn[1:] = d[1:] * (k[1:] / run)
    below = np.flatnonzero(dn[tauMin:] < YIN_TOL)
    with np.errstate(invalid="ignore", divide="ignore"):
        if len(below) == 0:
            m = np.abs(dn[tauMin:] - YIN_TOL) / YIN_TOL
            return 0, (float(np.min(m)) if np.isfinite(m).all() else math.inf), False
        first = tauMin + int(below[0])
        tau = first
        while tau + 1 < tauMax and dn[tau + 1] < dn[tau]:
            tau += 1
        margin = float(np.min(np.abs(dn[tauMin:first + 1] - YIN_TOL) / YIN_TOL))
        for j in range(first, min(tau, tauMax - 2) + 1):
            margin = min(margin, abs(dn[j + 1] - dn[j]) / max(abs(dn[j]), 1e-300))
    return tau, margin, first + 1 >= tauMax


# ---------------------------------------------------------------------------------------------------------------------
# input families: float32 [S][n] voices, one side chain, labels of the streams


def n_samples(fs, B, secs):
    return int(fs * secs) // B * B


def harmonic_voice(fs, n, seed, f0=None):
    """A sung vowel: three harmonics with vibrato and a little noise (seeded), peak below 0.8."""
    rng = np.random.default_rng(seed)
    f0 = rng.uniform(110.0, 320.0) if f0 is None else f0
    t = np.arange(n) / fs
    inst = f0 * (1.0 + 0.015 * np.sin(2 * np.pi * rng.uniform(4.0, 6.0) * t + rng.uniform(0.0, 2 * np.pi)))
    ph = 2 * np.pi * np.cumsum(inst) / fs
    x = (0.45 * np.sin(ph) + 0.22 * np.sin(2 * ph + rng.uniform(0.0, 2 * np.pi)) + 0.1 * np.sin(3 * ph + rng.uniform(0.0, 2 * np.pi))
         + 0.01 * rng.standard_normal(n))
    return x.astype(np.float32)


def side_chain(n):
    i = np.arange(n)
    return ((((3 * i) % 401) - 200) / 1024.0).astype(np.float32)  # the App. E side chain


def ladder_geometry(z, n):
    """Stretches of L + tauMax + 3 hopP samples, 2 stretch lengths of loud audio before, between and after them."""
    ls = z["win"] + 1 + 3 * z["hopP"]
    return list(range(ls, n - 2 * ls, 3 * ls)), ls


def ladder_family(fs, B, scales=LADDER, secs=2.0, voices=("kat", "harm")):
    """Each stream: a voice whose stretches are scaled by 2^-k (k = 140: FP32 subnormals), one stream per (voice, k)."""
    z = geom(fs, B)
    n = n_samples(fs, B, secs)
    starts, ls = ladder_geometry(z, n)
    base = {"kat": kat_inputs(int(fs), int(math.ceil(secs)))[0][:n], "harm": harmonic_voice(fs, n, 7)}
    rows, labels = [], []
    for name in voices:
        v = base[name]
        for k in scales:
            x = v.copy()
            for s0 in starts:
                x[s0:s0 + ls] = (v[s0:s0 + ls].astype(np.float64) * 2.0 ** -k).astype(np.float32)
            rows.append(x)
            labels.append({"voice": name, "k": k})
    return {"voice": np.array(rows), "labels": labels, "starts": starts, "ls": ls}


def dc_family(fs, B, per_case=DC_STREAMS, secs=1.0):
    """DC + a voice: d[k] = A + B - 2C cancels; the bound must send the frames of the heavy cases to FP64."""
    n = n_samples(fs, B, secs)
    rows, labels = [], []
    for ci, (dc, a) in enumerate(DC_CASES):
        for j in range(per_case):
            v = harmonic_voice(fs, n, 1000 + j).astype(np.float64)
            rows.append((dc + a * v).astype(np.float32))
            labels.append({"dc": dc, "a": a, "case": ci})
    return {"voice": np.array(rows), "labels": labels}


def _periodic_lambda(z, n, lam, per, noise):
    i = np.arange(n)
    return (per[i % len(per)] + lam * noise[i % len(noise)]).astype(np.float32)


def threshold_lambda(z):
    """Noise gain at which the dip's CMND of the steady-state frame crosses yinTol (bisection on the restatement)."""
    per, noise = _threshold_parts(z)
    n = 8 * z["hopP"] + z["win"]
    f = 6  # a frame whose window lies inside the input: every such frame sees the same samples (period hopP)
    w0 = f * z["hopP"] - z["latency"] - z["tauMax"]

    def dip(lam):
        x = _periodic_lambda(z, n, lam, per, noise)[w0:w0 + z["win"]]
        L, tauMin, tauMax = z["frameLenP"], z["tauMin"], z["tauMax"]
        xd = x.astype(np.float64)
        lagged = np.lib.stride_tricks.sliding_window_view(xd, L)[:tauMax]
        d = ((xd[:L] - lagged) ** 2).sum(axis=1)
        dn = d[1:] * (np.arange(1, tauMax) / np.cumsum(d[1:]))
        return float(dn[tauMin - 1:].min())
    lo, hi = 0.0, 0.05
    while dip(hi) < YIN_TOL:
        hi *= 2.0
    for _ in range(60):
        mid = 0.5 * (lo + hi)
        lo, hi = (mid, hi) if dip(mid) < YIN_TOL else (lo, mid)
    return 0.5 * (lo + hi)


def _threshold_parts(z):
    """A harmonic waveform of period chunk (= hopP / 3) and a noise sequence of period hopP: every frame that lies inside
    the input sees the same samples (frames start hopP apart), so one noise gain puts all of them at the same CMND."""
    T, hop = z["chunk"], z["hopP"]
    rng = np.random.default_rng(11)
    i = np.arange(T)
    per = sum(a * np.sin(2 * np.pi * h * i / T + rng.uniform(0.0, 2 * np.pi)) for h, a in ((1, 0.4), (2, 0.2), (3, 0.12), (4, 0.06)))
    return per, rng.standard_normal(hop) * 0.1


THRESHOLD_DELTAS = tuple(s * d for d in np.logspace(-1, -6, 11) for s in (-1.0, 1.0)) + (0.0,)


def threshold_family(fs, B, secs=1.0, deltas=THRESHOLD_DELTAS):
    z = geom(fs, B)
    n = n_samples(fs, B, secs)
    lam = threshold_lambda(z)
    per, noise = _threshold_parts(z)
    rows = [_periodic_lambda(z, n, lam * (1.0 + d), per, noise) for d in deltas]
    return {"voice": np.array(rows), "labels": [{"delta": d, "lambda": lam} for d in deltas]}


def edge_periods(z):
    tauMin, tauMax = z["tauMin"], z["tauMax"]
    exact = [239, 240, 241, tauMin, tauMin + 1, tauMax - 2, tauMax - 1]
    halves = [int(t) + 0.5 for t in np.linspace(tauMin + 1, tauMax - 2, 12).round()]
    return exact, halves


def edge_family(fs, B, secs=1.0):
    """Exact integer periods (a noise-like period tiled: d'(k) ~ 1 off the period, so the first lag under the threshold is
    the period itself) and harmonic voices of period T + 0.5 (d'(T) ~ d'(T + 1))."""
    z = geom(fs, B)
    n = n_samples(fs, B, secs)
    exact, halves = edge_periods(z)
    rng = np.random.default_rng(5)
    rows, labels = [], []
    for T in exact:
        seq = rng.uniform(-0.4, 0.4, T)
        rows.append(seq[np.arange(n) % T].astype(np.float32))
        labels.append({"period": T})
    t = np.arange(n)
    for P in halves:
        # (a little noise, as in a voice: three bare sinusoids leave the order-15 LPC of the pitch path singular)
        ph = 2 * np.pi * t / P
        rows.append((0.4 * np.sin(ph) + 0.2 * np.sin(2 * ph + 1.0) + 0.1 * np.sin(3 * ph + 2.0) + 0.01 * rng.standard_normal(n)).astype(np.float32))
        labels.append({"period": P})
    return {"voice": np.array(rows), "labels": labels}


BUILDERS = {"ladder": ladder_family, "dc": dc_family, "threshold": threshold_family, "edges": edge_family}
_INPUTS = {}


def family(name, rate, B=None):
    fs, B0 = RATES[rate]
    B = B or B0
    key = (name, rate, B)
    if key not in _INPUTS:
        fam = BUILDERS[name](fs, B)
        fam["synth"] = np.tile(side_chain(fam["voice"].shape[1]), (fam["voice"].shape[0], 1))
        fam["z"] = geom(fs, B)
        _INPUTS[key] = fam
    return _INPUTS[key]


def oracle_runs(fs, B, voice, synth, defined=False, params=None):
    """The C oracle on every stream (host threads; ctypes releases the GIL). The port, not the reference build: it defines
    what the reference leaves undefined at U3 (the descent ends at the last lag) and has the defined mode."""
    oraclebind.load()
    oraclebind.set_defined(defined)
    prm = params or {}
    try:
        with ThreadPoolExecutor(max_workers=max(1, len(os.sched_getaffinity(0)))) as ex:
            return list(ex.map(lambda s: oraclebind.run(fs, B, voice[s], synth[s], params=refbind.default_params(**prm), log=True),
                               range(len(voice))))
    finally:
        oraclebind.set_defined(False)


_ORACLE = {}


def family_oracle(name, rate, defined=False):
    key = (name, rate, defined)
    if key not in _ORACLE:
        fam = family(name, rate)
        _ORACLE[key] = oracle_runs(fam["z"]["fs"], fam["z"]["B"], fam["voice"], fam["synth"], defined=defined)
    return _ORACLE[key]


def inside_stretch_frames(fam, r):
    """Indices of the logged frames whose YIN window lies entirely inside one scaled stretch."""
    z, ls = fam["z"], fam["ls"]
    out = []
    for i, row in enumerate(r["pitch"]):
        _, w0 = frame_window(np.zeros(0), z, row)
        if any(s0 <= w0 and w0 + z["win"] <= s0 + ls for s0 in fam["starts"]):
            out.append(i)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# CPU tests


def _restatement_families(rate):
    """Small versions of every family (a few streams each) for the CPU checks."""
    fs, B = RATES[rate]
    dc = dc_family(fs, B, per_case=2)
    return {"ladder": ladder_family(fs, B, scales=(0, 66, 70, 75, 140), voices=("harm",)), "dc": dc,
            "threshold": threshold_family(fs, B, deltas=(-1e-2, -1e-5, 0.0, 1e-5, 1e-2)), "edges": edge_family(fs, B)}


@pytest.mark.parametrize("rate", sorted(RATES))
def test_restatement_gives_the_oracles_periods(rate):
    """yin64 decides every ungated frame of every family as the oracle does (frame positions from the oracle's log)."""
    fs, B = RATES[rate]
    z = geom(fs, B)
    for name, fam in _restatement_families(rate).items():
        synth = np.tile(side_chain(fam["voice"].shape[1]), (len(fam["voice"]), 1))
        refs = oracle_runs(fs, B, fam["voice"], synth, params=dict(vocBool=0))
        voiced = 0
        for s, r in enumerate(refs):
            assert len(r["pitch"]) == -(-fam["voice"].shape[1] // z["hopP"])
            for i, row in enumerate(r["pitch"]):
                if row.gated:
                    continue
                per, margin, u3 = yin64(frame_window(fam["voice"][s], z, row)[0], z)
                assert per == row.period, (name, fam["labels"][s], i, per, row.period, margin)
                voiced += per > 0
        assert voiced > 0, name


@pytest.mark.parametrize("rate", sorted(RATES))
def test_ladder_premise(rate):
    """Every stream of the ladder has frames that lie entirely inside a scaled stretch and are not gated (the ring the
    gate measures reaches loud audio next to the stretch), and the oracle gives those frames the periods of the unscaled
    voice: scaling by a power of two leaves the reference's CMND bit-identical. (The middle frames of a stretch are
    gated, so the first voiced frame after them has no previous marks: U4, flagged VP_PF_UB, lastMark = 0 on both sides.)"""
    fam = family("ladder", rate)
    refs = family_oracle("ladder", rate)
    z = fam["z"]
    for s, (lab, r) in enumerate(zip(fam["labels"], refs)):
        s0 = fam["labels"].index({"voice": lab["voice"], "k": 0})
        unscaled = refs[s0]["pitch"]
        idx = [i for i in inside_stretch_frames(fam, r) if not r["pitch"][i].gated]
        assert len(idx) >= LADDER_MIN_FRAMES, (lab, len(idx))
        exact = all(np.array_equal(fam["voice"][s][a:a + fam["ls"]].astype(np.float64) * 2.0 ** lab["k"],
                                   fam["voice"][s0][a:a + fam["ls"]].astype(np.float64)) for a in fam["starts"])
        assert exact or lab["k"] > 100, lab
        # (beyond 2^-100 the smallest samples are rounded to subnormals; these voices keep their periods all the same)
        assert [r["pitch"][i].period for i in idx] == [unscaled[i].period for i in idx], lab
        assert sum(r["pitch"][i].period > 0 for i in idx) >= LADDER_MIN_FRAMES // 2, lab  # voiced frames under test
    assert refs[0]["ub"] == 0 and z["tauMax"] > 0


@pytest.mark.parametrize("rate", sorted(RATES))
def test_threshold_premise(rate):
    """The noise gain puts the steady-state frames where the family says: within 10 delta (relative) of a decision,
    voiced below lambda*, unvoiced above it, and the frame at lambda* itself within 1e-9 of the threshold."""
    fam = family("threshold", rate)
    refs = family_oracle("threshold", rate)
    z = fam["z"]
    for s, (lab, r) in enumerate(zip(fam["labels"], refs)):
        res = {yin64(frame_window(fam["voice"][s], z, a)[0], z)[:2] for a in r["pitch"][4:10]}
        assert len(res) == 1, (lab, res)  # every steady-state frame sees the same samples
        (per, margin), = res
        assert per == r["pitch"][8].period, lab
        d = abs(lab["delta"])
        if d == 0.0:
            assert margin < 1e-9, margin
        elif d < 1e-2:
            assert margin < 10.0 * d and (per > 0) == (lab["delta"] < 0), (lab, per, margin)


def emulate_corr32(w, z):
    """C(k), k < tauMax, as k_yin_corr computes it: four chunk partials of c terms, each summed in FP32 in two levels
    (FFMA into a first-level sum, every YC_SUB terms -- groups of YC_R -- added to a second-level one) with gradual
    underflow; the partials added in double. The products of two floats are exact in double, so float32(p + acc) is the
    FFMA's single rounding (up to a double rounding, 2^-29 relative, far inside the bound's head room)."""
    L, c, tauMax = z["frameLenP"], z["chunk"], z["tauMax"]
    YC_R = 15
    x32 = np.asarray(w, np.float32)
    xd = x32.astype(np.float64)
    lagged = np.lib.stride_tricks.sliding_window_view(xd, L)[:tauMax].T  # [i][k] = x[i + k]
    tot = np.zeros(tauMax)
    for m in range(4):
        acc2 = np.zeros(tauMax, np.float32)
        acc = np.zeros(tauMax, np.float32)
        n = 0

        def ffma(j):
            return (xd[j] * lagged[j] + acc.astype(np.float64)).astype(np.float32)
        while n + YC_R <= c:
            n_sub = min(n + YC_SUB, c)
            while n + YC_R <= n_sub:
                for u in range(YC_R):
                    acc = ffma(m * c + n + u)
                n += YC_R
            acc2 = (acc2 + acc).astype(np.float32)
            acc = np.zeros(tauMax, np.float32)
        while n < c:
            acc = ffma(m * c + n)
            n += 1
        tot += (acc2 + acc).astype(np.float32).astype(np.float64)
    return tot


def corr_errors(w, z):
    """(|err d[k]|, relative bound, absolute term) per lag k >= 1 of the FP32 correlation form against float64."""
    L, tauMax = z["frameLenP"], z["tauMax"]
    xd = np.asarray(w, np.float32).astype(np.float64)
    lagged = np.lib.stride_tricks.sliding_window_view(xd, L)[:tauMax]
    A = float(np.dot(xd[:L], xd[:L]))
    Bk = (lagged ** 2).sum(axis=1)
    d_exact = ((xd[:L] - lagged) ** 2).sum(axis=1)
    d32 = (A + Bk) - 2.0 * emulate_corr32(w, z)
    err = np.abs(d32 - d_exact)[1:]
    rel = corr_beta(z["chunk"]) * (A + Bk[1:])
    return err, rel, np.where(A + Bk[1:] > 0.0, corr_abs(z["chunk"]), 0.0)


def test_corr_error_bound_holds_on_the_ladder_and_dc():
    """The FP32 correlation form stays within beta(c) (A + B(k)) plus the underflow term on every lag of ladder frames
    at every scale and of DC frames, and the purely relative bound does not: it fails once the products of the scaled
    samples reach the subnormal range (so the absolute term is what makes the bound rigorous there)."""
    for rate in ("44k", "96k"):
        fs, B = RATES[rate]
        z = geom(fs, B)
        lad = ladder_family(fs, B, voices=("harm",))
        n = lad["voice"].shape[1]
        s0 = lad["starts"][1]
        rel_fails = []
        for s, lab in enumerate(lad["labels"]):
            w = lad["voice"][s][s0:s0 + z["win"]]
            err, rel, ab = corr_errors(w, z)
            assert (err <= rel + ab).all(), (rate, lab, float(np.max(err / (rel + ab))))
            if (err > rel).any():
                rel_fails.append(lab["k"])
        assert rel_fails and min(rel_fails) <= 70 and 0 not in rel_fails and 60 not in rel_fails, rel_fails
        dc = dc_family(fs, B, per_case=1)
        for s, lab in enumerate(dc["labels"]):
            w = dc["voice"][s][3 * z["hopP"]:3 * z["hopP"] + z["win"]]
            err, rel, ab = corr_errors(w, z)
            assert (err <= rel + ab).all(), (rate, lab)
        assert n > 0


def test_all_zero_window_has_no_error_term():
    z = geom(44100.0, 1024)
    err, rel, ab = corr_errors(np.zeros(z["win"], np.float32), z)
    assert not err.any() and not rel.any() and not ab.any()


# ---------------------------------------------------------------------------------------------------------------------
# GPU tests


def set_path(monkeypatch, path):
    monkeypatch.delenv("VP_YIN_PHASES", raising=False)
    monkeypatch.delenv("VP_YIN_MODE", raising=False)
    if path == "single_pass":
        monkeypatch.setenv("VP_YIN_PHASES", "1")  # read at create
    elif path == "direct":
        monkeypatch.setenv("VP_YIN_MODE", "direct")  # read at prepare


def run_batch(vp, fam, mode=None):
    z = fam["z"]
    S, n = fam["voice"].shape
    eng = vp.Engine(z["fs"], z["B"], S, n // z["B"], params=vp.default_params())
    try:
        if mode is not None:
            eng.set_mode(mode)
        outL, _ = eng.process(fam["voice"], fam["synth"], None, want_right=False)
        frames = [eng.pitch_frames(s) for s in range(S)]
        st = eng.stats()
    finally:
        eng.close()
    return outL, frames, st


def check_streams(vp, fam, refs, outL, frames, what):
    """Stricter than assert_decisions: every frame without PF_NEAR_YIN | PF_NEAR_GATE | PF_UB matches the oracle exactly
    (gate, period, periodNew, note, marks, stale slot, beta), with no frames excused after a flagged one; a PF_NEAR_YIN
    frame must be within 1e-9 of a decision boundary by the float64 restatement; audio within the suite's tolerance.
    Returns the number of frames flagged PF_YIN_RECHECKED and the first mismatches."""
    z = fam["z"]
    skip = vp.PF_NEAR_YIN | vp.PF_NEAR_GATE | vp.PF_UB
    nre = 0
    bad = []
    for s, r in enumerate(refs):
        lab = fam["labels"][s]
        sn, mx = snr_db(r["outL"], outL[s]), maxabs(r["outL"], outL[s])
        assert sn >= SNR_MIN_DB and mx <= MAXABS_MAX, "%s %r: SNR %.1f dB, max abs err %.3e" % (what, lab, sn, mx)
        rows = oracle_decisions(r["pitch"])
        fr = frames[s]
        assert len(fr) == len(rows), (what, lab)
        for i, (a, b) in enumerate(zip(rows, fr)):
            if b.flags & vp.PF_YIN_RECHECKED:
                nre += 1
            if b.flags & vp.PF_NEAR_YIN:
                _, margin, _ = yin64(frame_window(fam["voice"][s], z, r["pitch"][i])[0], z)
                assert margin < 1e-9, (what, lab, i, margin)
            if b.flags & skip:
                continue
            gated = 1 if b.flags & vp.PF_GATED else 0
            ok = a["gated"] == gated
            if ok and not gated:
                ok = (a["period"] == b.period and a["note"] == b.note and a["an"] == list(b.anMarks[:b.nAn]) and
                      a["st"] == list(b.stMarks[:b.nSt]) and a["stale"] == b.anStale)
                if ok and a["an"]:
                    ok = a["periodNew"] == b.periodNew and a["beta"] == b.beta
            if not ok:
                bad.append("%r frame %d: oracle gated=%d period=%d note=%d | engine flags=%d period=%d note=%d" % (
                    lab, i, a["gated"], a["period"], a["note"], b.flags, b.period, b.note))
    assert not bad, "%s: %d frames differ from the oracle, first: %s" % (what, len(bad), "; ".join(bad[:6]))
    return nre


@pytest.mark.gpu
@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("rate", sorted(RATES))
@pytest.mark.parametrize("name", FAMILIES)
def test_family_matches_oracle(vp, monkeypatch, name, rate, path):
    fam = family(name, rate)
    refs = family_oracle(name, rate)
    set_path(monkeypatch, path)
    outL, frames, st = run_batch(vp, fam)
    what = "%s %s %s" % (name, rate, path)
    nre = check_streams(vp, fam, refs, outL, frames, what)
    assert st["yin_rechecked"] == nre, (what, st["yin_rechecked"], nre)
    z = fam["z"]
    if name == "dc" and path != "direct":
        # the heaviest cancellation: the bound cannot resolve these frames in FP32, they are decided in FP64
        heavy = [s for s, lab in enumerate(fam["labels"]) if lab["case"] == len(DC_CASES) - 1]
        voiced = [(s, i) for s in heavy for i, a in enumerate(refs[s]["pitch"]) if a.period > 0]
        re = sum(1 for s, i in voiced if frames[s][i].flags & vp.PF_YIN_RECHECKED)
        assert len(heavy) >= 128 and len(voiced) > 0.5 * sum(len(refs[s]["pitch"]) for s in heavy)
        assert re >= 0.9 * len(voiced), (what, re, len(voiced))
    if name == "edges":
        # U3 (the descent starts at tauMax - 1): the engine says where the reference is undefined
        s = fam["labels"].index({"period": z["tauMax"] - 1})
        u3 = [i for i, a in enumerate(refs[s]["pitch"]) if not a.gated and yin64(frame_window(fam["voice"][s], z, a)[0], z)[2]]
        assert len(u3) > 0.5 * len(refs[s]["pitch"]) and refs[s]["ub"] & 2
        assert all(frames[s][i].flags & vp.PF_UB for i in u3), what
    if name == "threshold":
        # both sides of yinTol are reached: voiced and unvoiced steady-state frames
        per = [frames[s][8].period for s in range(len(frames))]
        assert min(per) == 0 and max(per) > 0, per


@pytest.mark.gpu
@pytest.mark.parametrize("rate", ("44k", "48k"))
@pytest.mark.parametrize("name", FAMILIES)
def test_two_phase_equals_single_pass(vp, monkeypatch, name, rate):
    """The two lag phases and one pass over all lags give bit-identical periods, marks, flags and audio on every family.
    (Which frames go to FP64 may differ: phase 1 checks the lags below the split only.)"""
    fam = family(name, rate)
    res = []
    for path in ("two_phase", "single_pass"):
        set_path(monkeypatch, path)
        outL, frames, _ = run_batch(vp, fam)
        res.append((outL, [[(f.flags & ~vp.PF_YIN_RECHECKED, f.period, f.note, list(f.anMarks[:f.nAn]), list(f.stMarks[:f.nSt]))
                            for f in fr] for fr in frames]))
    assert res[0][1] == res[1][1]
    assert np.array_equal(res[0][0], res[1][0])


@pytest.mark.gpu
@pytest.mark.parametrize("rate", sorted(RATES))
def test_edge_lags_in_defined_mode(vp, monkeypatch, rate):
    """VP_MODE_DEFINED on the edge lags: the descent ends at the last lag where the reference reads yinTemp[tauMax]; the
    engine matches the oracle's defined mode and flags nothing as undefined."""
    fam = family("edges", rate)
    refs = family_oracle("edges", rate, defined=True)
    set_path(monkeypatch, "two_phase")
    outL, frames, st = run_batch(vp, fam, mode=vp.VP_MODE_DEFINED)
    nre = check_streams(vp, fam, refs, outL, frames, "edges %s defined" % rate)
    assert st["yin_rechecked"] == nre
    assert not any(f.flags & vp.PF_UB for fr in frames for f in fr)
    s = fam["labels"].index({"period": fam["z"]["tauMax"] - 1})
    assert sum(f.period == fam["z"]["tauMax"] - 1 for f in frames[s]) > 0.5 * len(frames[s])


@pytest.mark.gpu
def test_ladder_streaming_blocks(vp, monkeypatch):
    """The ladder through vp_engine_stream_block at B = 128: one pitch frame per block at most, single-phase decision."""
    fs, B = 44100.0, 128
    fam = ladder_family(fs, B, scales=(0, 68, 75, 140), voices=("harm",))
    fam["synth"] = np.tile(side_chain(fam["voice"].shape[1]), (len(fam["voice"]), 1))
    fam["z"] = geom(fs, B)
    refs = oracle_runs(fs, B, fam["voice"], fam["synth"])
    set_path(monkeypatch, "two_phase")
    S, n = fam["voice"].shape
    eng = vp.Engine(fs, B, S, 1, params=vp.default_params())
    try:
        hv, hs, ho = eng.stream_buffers()
        out = np.zeros((S, n), np.float32)
        frames = [[] for _ in range(S)]
        nst = 0
        for b in range(n // B):
            hv[:] = fam["voice"][:, b * B:(b + 1) * B]
            hs[:] = fam["synth"][:, b * B:(b + 1) * B]
            eng.stream_block()
            out[:, b * B:(b + 1) * B] = ho
            for s in range(S):
                frames[s] += eng.pitch_frames(s)
            nst += eng.stats()["yin_rechecked"]
    finally:
        eng.close()
    nre = check_streams(vp, fam, refs, out, frames, "ladder streaming B=128")
    assert nst == nre
