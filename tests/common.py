"""Shared helpers of the parity tests: the SURVEY App. E known-answer inputs,
error metrics, decision comparison, golden-fixture access."""
import hashlib
import json
import os
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")

# Stated tolerances of BASELINE.json's north_star (audio vs the float32 reference).
SNR_MIN_DB = 80.0
MAXABS_MAX = 1e-4


def kat_inputs(fs=44100, seconds=4):
    """SURVEY.md App. E: integer-arithmetic inputs, exactly representable in float32."""
    n = seconds * fs
    x = 12345
    noise = np.empty(n)
    for i in range(n):
        x = (1664525 * x + 1013904223) & 0xFFFFFFFF
        noise[i] = ((x >> 16) - 32768) / 2.0 ** 22
    i = np.arange(n)
    voice = (((i % 221) - 110) / 256.0 + noise).astype(np.float32)
    synth = ((((3 * i) % 401) - 200) / 1024.0).astype(np.float32)
    return voice, synth


def snr_db(ref, x):
    ref = np.asarray(ref, np.float64)
    x = np.asarray(x, np.float64)
    err = float(np.sum((ref - x) ** 2))
    sig = float(np.sum(ref ** 2))
    if err == 0.0:
        return 300.0
    if sig == 0.0:
        return -300.0
    return 10.0 * np.log10(sig / err)


def maxabs(ref, x):
    return float(np.max(np.abs(np.asarray(ref, np.float64) - np.asarray(x, np.float64)))) if len(ref) else 0.0


def crc(a):
    return "%08x" % zlib.crc32(np.ascontiguousarray(a).tobytes())


def stats(out):
    o = np.asarray(out, np.float64)
    nz = np.flatnonzero(o)
    return {"first_nonzero": int(nz[0]) if len(nz) else -1, "sum": float(o.sum()), "sum_abs": float(np.abs(o).sum()),
            "rms": float(np.sqrt(np.mean(o * o))), "max_abs": float(np.abs(o).max())}


def oracle_decisions(plog):
    """Per pitch frame decisions of an oracle / reference log as plain tuples."""
    rows = []
    for a in plog:
        rows.append({"gated": int(a.gated), "period": int(a.period), "periodNew": int(a.periodNew), "note": int(a.note),
                     "an": [int(v) for v in a.anMarks[:a.nAn]], "st": [int(v) for v in a.stMarks[:a.nSt]],
                     "stale": int(a.anStale), "beta": float(a.beta)})
    return rows


class Decisions(tuple):
    """(n, bad, flagged, first, checked, excused) of compare_decisions; fields by name as well."""
    __slots__ = ()
    _names = ("n", "bad", "flagged", "first", "checked", "excused")

    def __new__(cls, *vals):
        return tuple.__new__(cls, vals)

    def __getattr__(self, k):
        try:
            return self[self._names.index(k)]
        except ValueError:
            raise AttributeError(k)


RESYNC_FRAMES = 2     # agreeing frames after a flagged one before the comparison is trusted again
PROBATION_FRAMES = 8  # frames after such a re-synchronisation in which a difference re-opens the excused stretch


def compare_decisions(vp, ref_rows, eng_frames):
    """Bit-exact comparison of the integer decisions (period, snapped note, marks) of one stream.

    Returns Decisions(n, bad, flagged, first, checked, excused):
      n        frames present on both sides,
      flagged  frames the engine flags as within epsilon of a decision boundary, or as undefined behaviour in the
               reference (not compared: the reference's own answer is not authoritative there),
      checked  frames compared AND counted: every caller asserts checked >= CHECKED_FLOOR * n, so a test cannot pass
               with most of a stream unchecked,
      bad      compared frames that differ,
      excused  frames after a flagged one that differ before the two mark chains agree again (the chain carries state
               from frame to frame; once RESYNC_FRAMES consecutive frames agree in every field the comparison resumes),
      first    text of the first mismatch."""
    n = min(len(ref_rows), len(eng_frames))
    bad = flagged = checked = excused = 0
    first = None
    taint = probation = 0
    for i in range(n):
        a, b = ref_rows[i], eng_frames[i]
        if b.flags & (vp.PF_NEAR_YIN | vp.PF_NEAR_GATE | vp.PF_UB):
            flagged += 1
            taint = RESYNC_FRAMES
            continue
        gated = 1 if (b.flags & vp.PF_GATED) else 0
        ok = a["gated"] == gated
        if ok and not gated:
            ok = (a["period"] == b.period and a["an"] == list(b.anMarks[:b.nAn]) and a["st"] == list(b.stMarks[:b.nSt]) and
                  a["note"] == b.note and a["stale"] == b.anStale)
            if ok and a["an"]:
                ok = a["periodNew"] == b.periodNew and a["beta"] == b.beta
        if taint > 0:
            if ok:
                taint -= 1
                checked += 1
                if taint == 0:
                    probation = PROBATION_FRAMES
            else:
                excused += 1
                taint = RESYNC_FRAMES
            continue
        if not ok and probation > 0:
            excused += 1
            taint = RESYNC_FRAMES
            probation = 0
            continue
        probation = max(0, probation - 1)
        checked += 1
        if not ok:
            bad += 1
            if first is None:
                first = "frame %d ref %r | eng flags=%d period=%d pnew=%d note=%d an=%r st=%r stale=%d beta=%r" % (
                    i, a, b.flags, b.period, b.periodNew, b.note, list(b.anMarks[:b.nAn]), list(b.stMarks[:b.nSt]),
                    b.anStale, b.beta)
    return Decisions(n, bad, flagged, first, checked, excused)


CHECKED_FLOOR = 0.98


def assert_decisions(dec, what=""):
    """0 mismatches and at least CHECKED_FLOOR of the frames actually compared."""
    assert dec.bad == 0, "%s: %s" % (what, dec.first)
    assert dec.checked >= CHECKED_FLOOR * dec.n, "%s: only %d of %d frames compared (%d flagged, %d excused)" % (
        what, dec.checked, dec.n, dec.flagged, dec.excused)


def golden_index():
    with open(os.path.join(GOLDEN, "index.json")) as f:
        return json.load(f)


def golden_load(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def sha256(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def reference_pin(r):
    """A run of the reference (or of the oracle) in the form tests/golden/reference_build_pins.json stores it: both output
    channels by SHA-256 of their float bytes, the sizes, and every pitch decision in full."""
    return {"outL_sha256": sha256(r["outL"]), "outR_sha256": sha256(r["outR"]), "n": int(len(r["outL"])),
            "sizes": r["sizes"], "decisions": oracle_decisions(r["pitch"])}


def reference_pins():
    with open(os.path.join(GOLDEN, "reference_build_pins.json")) as f:
        return json.load(f)


def reference_runs(jobs, threads=None):
    """Runs the CPU reference on many streams at once (host threads; ctypes releases the GIL).
    jobs: [(fs, B, voice, synthL, synthR or None, params dict)]. Uses oracle/_ref (the reference's own C++) when it is
    built on this machine, else the C oracle port (bit-identical to it, tests/test_oracle.py). Returns (results, kind)."""
    import os
    from concurrent.futures import ThreadPoolExecutor
    import oraclebind
    import refbind
    use_ref = refbind.available("strict")
    if not use_ref:
        oraclebind.load()

    def one(job):
        fs, B, v, l, r, params = job
        prm = refbind.default_params(**params)
        if use_ref:
            return refbind.run(fs, B, v, l, synthR=r, params=prm, log=True)
        return oraclebind.run(fs, B, v, l, synthR=r, params=prm, log=True)
    threads = threads or max(1, len(os.sched_getaffinity(0)))
    with ThreadPoolExecutor(max_workers=threads) as ex:
        res = list(ex.map(one, jobs))
    return res, ("reference" if use_ref else "port")
