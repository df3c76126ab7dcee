#!/usr/bin/env python
"""bench.py -- throughput of the hot path (VocoderProject DSP core, batched over streams).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl engine|reference] [--workload NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch of synthetic streams: per stream it is
equivalent to prepareToPlay + nBlocks processBlock calls of the reference plug-in
(PluginProcessor.cpp:144-234). Metric: audio-seconds processed per second (x real-time,
summed over streams and GPUs). Streams shard by contiguous ranges over ranks with NO
data-path collective (weak scaling: the per-GPU batch is fixed).

One JSON line on stdout (rank 0). `value`: inputs resident in HBM, device time (CUDA events
on the engine's stream, max over ranks). `e2e`: the same batch through the C-ABI host call
vp_engine_process_host with pinned HOST buffers (H2D + compute + D2H inside the timed region).
`--impl reference`: the reference's own C++ (oracle/_ref, compiled in place; else the C oracle
port) on the host cores, on a bounded sample of the same workload.
`--dump-outputs DIR`: after the timed steps, a fixed, seeded sample (at most 64 MB) of the audio the last timed step
returned, as DIR/outL_rows.npy and DIR/outL_cols.npy (float32). The inputs are seeded too, so two builds run with the
same arguments can be compared output for output.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

# workloads: SURVEY.md 8(d) / BASELINE.json configs. Per-GPU stream counts (weak scaling).
WORKLOADS = {
    # configs[3]: full chain, 16384 streams x 60 s @ 48 kHz over 8 GPUs = 2048 streams per GPU
    "chain48": dict(desc="full vocoder + pitch-corrector chain, 2048 streams/GPU x 60 s @ 48 kHz, chromatic, block 1024 "
                         "(BASELINE configs[3] = 16384 streams over 8 GPUs)",
                    fs=48000.0, B=1024, seconds=60.0, streams=2048, params=dict()),
    # configs[1]: vocoder only, 1024 pairs x 30 s @ 44.1 kHz
    "voc44": dict(desc="vocoder only, 1024 voice/carrier pairs x 30 s @ 44.1 kHz, LPC 40/5 (BASELINE configs[1])",
                  fs=44100.0, B=1024, seconds=30.0, streams=1024, params=dict(pitchBool=0)),
    # configs[2]: pitch corrector only, 4096 streams x 30 s @ 44.1 kHz, chromatic
    "pitch44": dict(desc="pitch corrector only, 4096 streams x 30 s @ 44.1 kHz, chromatic (BASELINE configs[2])",
                    fs=44100.0, B=1024, seconds=30.0, streams=4096, params=dict(vocBool=0)),
    # the north_star target line: chain at 44.1 kHz
    "chain44": dict(desc="full chain, 2048 streams/GPU x 60 s @ 44.1 kHz, chromatic, block 1024",
                    fs=44100.0, B=1024, seconds=60.0, streams=2048, params=dict()),
    "tiny": dict(desc="smoke-size chain, 64 streams x 4 s @ 44.1 kHz", fs=44100.0, B=1024, seconds=4.0, streams=64,
                 params=dict()),
}

# Algorithmic FP32 lane-operations ("slots": one FADD/FMUL/FFMA each) per frame, minimal direct
# form, SURVEY.md App. C.5 -- the denominators of the roofline fractions (DESIGN.md section 5).


def slot_model(sz, prm):
    wl, hopV, L, hopP, c, tauMax = sz["wlenV"], sz["hopV"], sz["frameLenP"], sz["hopP"], sz["chunk"], sz["tauMax"]
    pv, ps, pp = prm.lpcVoice, prm.lpcSynth, prm.lpcPitch

    def ac(n, p):  # windowed autocorrelation, lags 0..p
        return sum(n - m for m in range(p + 1))

    def lev(p):
        return sum(2 * (q - 1) + 2 + q for q in range(2, p + 1)) + 1 + p

    def fir(n, p):
        return sum(min(i, p) + 1 for i in range(n))

    voc = {"window": 2 * wl, "autocorr_voice": ac(wl, pv), "autocorr_synth": ac(wl, ps), "levinson": lev(pv) + lev(ps),
           "fir_voice": fir(wl, pv) + wl, "fir_synth": fir(wl, ps) + wl, "gain": 22, "iir": fir(wl, pv) - wl + wl, "ola": wl}
    keepNeeded = tauMax
    pitch = {"yin": 2 * L * tauMax, "cmnd": 3 * tauMax, "autocorr": ac(L, pp), "levinson": lev(pp),
             "residual_fir": (keepNeeded + L + 3 * c) * (pp + 1), "psola": 12 * L, "iir": fir(L, pp), "ola": L}
    return {"voc_per_frame": sum(voc.values()), "pitch_per_frame": sum(pitch.values()), "voc": voc, "pitch": pitch,
            "voc_per_sample": sum(voc.values()) / hopV, "pitch_per_sample": sum(pitch.values()) / hopP}


def mix_capture(workload):
    """Executed FP64 / FP32 thread-instructions and DRAM bytes per audio sample of every stage, from the newest committed
    ncu capture (profiles/ncu_mix_*.json, tools/ncu_mix.py). None when there is none for this workload."""
    import glob
    try:
        with open(sorted(glob.glob(os.path.join(ROOT, "profiles", "ncu_mix_*.json")))[-1]) as f:
            mj = json.load(f)
        w = mj["workloads"].get(workload)
        if w:
            w = dict(w, source=mj["source"])
        return w
    except Exception:
        return None


def mix_roofline(workload, samples_per_step, ms_per_step, peaks_fp, sm_mhz, n_sm=148):
    """Instruction-mix roofline of a step: the FP64 and FP32 arithmetic instructions the kernels EXECUTE (ncu), each at the
    issue rate of its pipe. A DFMA holds the SM sub-partition's dispatch port for two cycles and nothing else issues next to
    it (profiles/ubench_mix_r02a.txt), so the two terms add: lower_bound = fp64_ops / fp64_rate + fp32_ops / fp32_rate."""
    w = mix_capture(workload)
    if not w:
        return None
    f64, f32 = w["total"]["fp64_ops_per_sample"], w["total"]["fp32_ops_per_sample"]
    p64, p32 = peaks_fp["fp64_fma_per_s"], peaks_fp["fp32_fma_per_s"]
    lb_ms = 1e3 * samples_per_step * (f64 / p64 + f32 / p32)
    clk = (sm_mhz or 1965.0) * 1e6
    th64, th32 = n_sm * 64 * clk, n_sm * 128 * clk
    lb_th = 1e3 * samples_per_step * (f64 / th64 + f32 / th32)
    return {"fp64_ops_per_sample": f64, "fp32_ops_per_sample": f32, "thread_inst_per_sample": w["total"]["thread_inst_per_sample"],
            "dram_bytes_per_sample": w["total"]["dram_bytes_per_sample"], "lower_bound_ms": lb_ms, "ms_per_step": ms_per_step,
            "frac": lb_ms / ms_per_step if ms_per_step else None,
            "lower_bound_ms_theoretical_rates": lb_th, "frac_theoretical_rates": lb_th / ms_per_step if ms_per_step else None,
            "issue_rates_per_s": {"fp64_measured": p64, "fp32_measured": p32, "fp64_theoretical": th64, "fp32_theoretical": th32,
                                  "theoretical": "%d SMs x 64 (FP64) / 128 (FP32) lanes x %.0f MHz" % (n_sm, clk / 1e6)},
            "per_stage": {k: {"fp64": round(v["fp64_ops_per_sample"], 2), "fp32": round(v["fp32_ops_per_sample"], 2),
                              "dram_bytes": round(v["dram_bytes_per_sample"], 2)} for k, v in w["stages"].items()},
            "source": w["source"], "note": "executed arithmetic thread-instructions per audio sample (ncu, %d samples per captured pass) x samples "
                                           "of a step; DADD / DMUL / FADD / FMUL count like an FMA of their pipe" % w["samples_per_pass_capture"]}


DUMP_BYTES = 64 << 20   # --dump-outputs writes at most this much in all


def dump_sample(read_row, S, n, budget=DUMP_BYTES, seed=0):
    """A fixed, seeded sample of a float32 [S][n] output that read_row(s) returns one row at a time, in two arrays of at most
    budget / 2 bytes each: "rows", a few whole streams (a seeded window of each when a stream alone is larger), and
    "cols", every stream at a few seeded sample positions. The sample depends on (S, n, budget, seed) only, so that runs
    of two builds with the same arguments can be compared value for value. Returns ({name: array}, {what was sampled})."""
    rng = np.random.default_rng(seed)
    half = budget // 2 // 4
    L = min(n, half)
    streams = np.sort(rng.choice(S, size=max(1, min(S, half // L)), replace=False))
    off = int(rng.integers(0, n - L + 1))
    cols = np.sort(rng.choice(n, size=max(1, min(n, half // S)), replace=False))
    rows = np.empty((len(streams), L), np.float32)
    at = np.empty((S, len(cols)), np.float32)
    for s in range(S):
        row = read_row(s)
        at[s] = row[cols]
        k = np.searchsorted(streams, s)
        if k < len(streams) and streams[k] == s:
            rows[k] = row[off:off + L]
    return {"rows": rows, "cols": at}, {"streams": streams.tolist(), "row_offset": off, "row_length": L, "cols": len(cols),
                                        "seed": seed}


def dump_outputs(eng, do, S, n, group, out_dir):
    """--dump-outputs: writes a sample of what the last timed step left in the output buffer `do` (outL, float32 [S][n] on
    the device) as out_dir/outL_rows.npy and out_dir/outL_cols.npy (see dump_sample); with several ranks each writes its
    own shard's sample as rank<r>_outL_*.npy, and the ranks share the size budget."""
    def read_row(s):
        row = np.empty(n, np.float32)
        eng._check(eng.lib.vp_memcpy_d2h(eng.h, row.ctypes.data, C.c_void_p(do + s * n * 4), n * 4))
        return row
    arrays, what = dump_sample(read_row, S, n, budget=DUMP_BYTES // group.world)
    os.makedirs(out_dir, exist_ok=True)
    prefix = "rank%d_" % group.rank if group.world > 1 else ""
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, "%soutL_%s.npy" % (prefix, k)), a)
    return dict(what, dir=out_dir, arrays={prefix + "outL_" + k: list(a.shape) for k, a in arrays.items()})


def run_sub(vp, args, name, group, peaks_fp, sm_mhz):
    """Short device-resident run of another BASELINE configuration (--warmup and --steps as given), for the result line's
    other_workloads."""
    wl = WORKLOADS[name]
    fs, B = wl["fs"], wl["B"]
    n = int(fs * wl["seconds"]) // B * B
    S = wl["streams"]
    prm = vp.default_params(**wl["params"])
    eng = vp.Engine(fs, B, S, n // B, params=prm, device=group.local_rank)
    try:
        nb = S * n * 4
        dv, dl, do = eng.device_alloc(nb), eng.device_alloc(nb), eng.device_alloc(nb)
        eng.synth_device(0, group.rank * S, S, n, n, dv, dl, None)
        for _ in range(args.warmup):
            eng.reset()
            eng.process_device(n // B, dv, dl, None, do, None, n, sync=False)
        eng.sync()
        steps = args.steps
        eng.timer_record(0)
        for _ in range(steps):
            eng.reset()
            eng.process_device(n // B, dv, dl, None, do, None, n, sync=False)
        eng.timer_record(1)
        eng.sync()
        sec = eng.timer_elapsed_ms(0, 1) * 1e-3
        sm = slot_model(eng.sizes, prm)
        slots = (sm["voc_per_sample"] if prm.vocBool else 0.0) + (sm["pitch_per_sample"] if prm.pitchBool else 0.0)
        ms = 1e3 * sec / steps
        res = {"workload": wl["desc"], "value": S * n / fs * steps / sec, "unit": "audio-s/s", "ms_per_step": ms, "steps": steps, "warmup": args.warmup,
               "streams": S, "seconds_per_stream": n / fs,
               "chain_frac": slots * S * n * steps / sec / peaks_fp["fp32_fma_per_s"], "slots_per_sample": slots}
        mx = mix_roofline(name, float(S) * n, ms, peaks_fp, sm_mhz)
        if mx:
            res["mix_frac"] = mx["frac"]
            res["mix_lower_bound_ms"] = mx["lower_bound_ms"]
        for p_ in (dv, dl, do):
            eng.device_free(p_)
        return res
    finally:
        eng.close()


class ClockSampler:
    """nvidia-smi clocks + throttle reasons of one GPU, sampled every 200 ms while running."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.th = [], None, None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def window(self, t0, t1):
        rows = [r for t, r in self.rows if t0 <= t <= t1] or [r for _, r in self.rows[-1:]]
        sm, mx, reasons, pw = [], [], set(), []
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm),
                "reasons": sorted(reasons)}

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


def numa_bind(dev_index):
    """Binds this process to the CPUs of the NUMA node the GPU hangs off (pinned buffers are then allocated, first touch, on
    that node: a copy does not cross the inter-socket link). Returns a description for the JSON line."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(dev_index), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip())
        nodes = [d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()]
        if node < 0 or len(nodes) < 2:
            return {"gpu_numa_node": node, "nodes": len(nodes), "bound": False}
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus |= set(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return {"gpu_numa_node": node, "nodes": len(nodes), "bound": False}
        os.sched_setaffinity(0, cpus)
        return {"gpu_numa_node": node, "nodes": len(nodes), "bound": True, "cpus": len(cpus)}
    except Exception as ex:
        return {"bound": False, "error": str(ex)[:80]}


def link_ceiling(n_gpus):
    """Pinned-copy rates of the host link with n_gpus GPUs copying at once, from the newest committed probe log that covers
    n_gpus (tools/link_probe.cu -> profiles/link_probe_*.jsonl): H2D alone, D2H alone, and both directions at once (total).
    None when no log covers n_gpus."""
    import glob
    best = None
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "link_probe_*.jsonl"))):
        got = {}
        for ln in open(path):
            try:
                j = json.loads(ln)
            except ValueError:
                continue
            if j.get("gpus") != n_gpus or j.get("copy") != "1d" or j.get("pinned") != "default" or j.get("numa_bound"):
                continue
            if j.get("h2d") and j.get("d2h"):
                got["duplex"] = max(got.get("duplex", 0.0), j["duplex_gbs_total"])
            elif j.get("h2d"):
                got["h2d"] = max(got.get("h2d", 0.0), j["h2d_gbs_total"])
            elif j.get("d2h"):
                got["d2h"] = max(got.get("d2h", 0.0), j["d2h_gbs_total"])
        if len(got) == 3:
            best = dict(got, file=path)
    return best


def live_link_probe(group, dev, h_src, h_dst, nbytes, reps=4):
    """The same three rates measured on THIS box inside the run (tools/link_probe.cu's method through libcudart): every rank
    copies `nbytes` of the pinned end-to-end buffers up / down / both ways on two streams, all ranks released together by a
    barrier; rates are summed over the ranks. The committed probe logs describe the boxes they were taken on -- a 2-GPU box is
    not the first two GPUs of an 8-GPU box. Returns None when the runtime library cannot be loaded or a call fails on any
    rank; every rank makes the same collective calls whatever happens locally."""
    vpp, sz = C.c_void_p, C.c_size_t
    rt = None
    d_in, d_out, s_a, s_b = vpp(), vpp(), vpp(), vpp()
    ev = [vpp() for _ in range(4)]

    def ok(rc):
        if rc != 0:
            raise RuntimeError("cudart call failed: %d" % rc)

    good = True
    try:
        for name in ("libcudart.so.12", "libcudart.so", "/usr/local/cuda/lib64/libcudart.so"):
            try:
                rt = C.CDLL(name)
                break
            except OSError:
                continue
        if rt is None:
            raise RuntimeError("libcudart not found")
        rt.cudaMalloc.argtypes = [C.POINTER(vpp), sz]
        rt.cudaFree.argtypes = [vpp]
        rt.cudaStreamCreateWithFlags.argtypes = [C.POINTER(vpp), C.c_uint]
        rt.cudaStreamDestroy.argtypes = [vpp]
        rt.cudaEventCreate.argtypes = [C.POINTER(vpp)]
        rt.cudaEventDestroy.argtypes = [vpp]
        rt.cudaEventRecord.argtypes = [vpp, vpp]
        rt.cudaEventElapsedTime.argtypes = [C.POINTER(C.c_float), vpp, vpp]
        rt.cudaMemcpyAsync.argtypes = [vpp, vpp, sz, C.c_int, vpp]
        rt.cudaStreamSynchronize.argtypes = [vpp]
        ok(rt.cudaSetDevice(C.c_int(dev)))
        ok(rt.cudaMalloc(C.byref(d_in), nbytes))
        ok(rt.cudaMalloc(C.byref(d_out), nbytes))
        ok(rt.cudaStreamCreateWithFlags(C.byref(s_a), 1))
        ok(rt.cudaStreamCreateWithFlags(C.byref(s_b), 1))
        for e_ in ev:
            ok(rt.cudaEventCreate(C.byref(e_)))
    except Exception as ex:
        sys.stderr.write("live link probe: set-up failed: %r\n" % (ex,))
        good = False
    good = group.min(1.0 if good else 0.0) > 0.5   # all ranks or none

    def issue(up, down):
        if up:
            ok(rt.cudaMemcpyAsync(d_in, vpp(h_src), nbytes, 1, s_a))
        if down:
            ok(rt.cudaMemcpyAsync(vpp(h_dst), d_out, nbytes, 2, s_b))

    out = {"file": None, "live_gib": nbytes / 2.0**30}
    if good:
        for key, up, down in (("h2d", True, False), ("d2h", False, True), ("duplex", True, True)):
            rate, failed = 0.0, False
            try:
                issue(up, down)
                ok(rt.cudaStreamSynchronize(s_a)); ok(rt.cudaStreamSynchronize(s_b))
            except Exception:
                failed = True
            group.barrier()
            try:
                if not failed:
                    ok(rt.cudaEventRecord(ev[0], s_a)); ok(rt.cudaEventRecord(ev[2], s_b))
                    for _ in range(reps):
                        issue(up, down)
                    ok(rt.cudaEventRecord(ev[1], s_a)); ok(rt.cudaEventRecord(ev[3], s_b))
                    ok(rt.cudaStreamSynchronize(s_a)); ok(rt.cudaStreamSynchronize(s_b))
                    for on, e0, e1 in ((up, ev[0], ev[1]), (down, ev[2], ev[3])):
                        if on:
                            ms = C.c_float()
                            ok(rt.cudaEventElapsedTime(C.byref(ms), e0, e1))
                            rate += reps * nbytes / (ms.value * 1e-3) / 1e9
            except Exception as ex:
                sys.stderr.write("live link probe: %s failed: %r\n" % (key, ex))
                failed = True
            out[key] = group.sum(rate)
            if group.max(1.0 if failed else 0.0) > 0.5:
                good = False
    if rt is not None:
        try:
            for e_ in ev:
                if e_.value:
                    rt.cudaEventDestroy(e_)
            if s_a.value:
                rt.cudaStreamDestroy(s_a)
            if s_b.value:
                rt.cudaStreamDestroy(s_b)
            if d_in.value:
                rt.cudaFree(d_in)
            if d_out.value:
                rt.cudaFree(d_out)
        except Exception:
            pass
    return out if good and all(out.get(k_, 0) > 0 for k_ in ("h2d", "d2h", "duplex")) else None


def link_bound(link, h2d_bytes, d2h_bytes):
    """Time (s) the host link needs at least for a step's copies: each direction at its rate when it runs alone, and both
    together at the total rate measured with both directions busy (the host's memory system is shared: with 8 GPUs the
    duplex total, 159 GB/s, is far below the sum of the one-way rates, 236 + 119 GB/s)."""
    return max(h2d_bytes / (link["h2d"] * 1e9), d2h_bytes / (link["d2h"] * 1e9), (h2d_bytes + d2h_bytes) / (link["duplex"] * 1e9))


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_run(kind_pref, fs, B, voice, sl, params_kw, threads):
    """One pass of the reference CPU path over [S][n] host arrays. Returns (seconds, kind)."""
    import oraclebind
    import refbind
    prm = refbind.default_params(**params_kw)
    if kind_pref == "reference" and refbind.available("fast"):
        sec, _ = refbind.bench(fs, B, voice, sl, None, params=prm, threads=threads, kind="fast")
        return sec, "reference"
    sec, _ = oraclebind.bench(fs, B, voice, sl, None, params=prm, threads=threads)
    return sec, "port"


def gen_host_inputs(vp, fs, first, S, n, threads):
    """vp_synth_host over `threads` Python threads (ctypes releases the GIL). vp = None: the stand-alone generator
    tools/_build/libvp_inputgen.so (same definitions, no CUDA, no product library in the process)."""
    voice = np.zeros((S, n), np.float32)
    sl = np.zeros((S, n), np.float32)
    if vp is None:
        fn = C.CDLL(os.path.join(ROOT, "tools", "_build", "libvp_inputgen.so")).vpgen_synth_host
        fn.restype = C.c_int
        fn.argtypes = [C.c_double, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]
    else:
        fn = vp.load_library().vp_synth_host

    def work(t):
        for s in range(t, S, threads):
            fn(float(fs), 0, first + s, 1, n, n, voice[s].ctypes.data, sl[s].ctypes.data, None)
    ths = [threading.Thread(target=work, args=(t,)) for t in range(min(threads, S))]
    [t.start() for t in ths]
    [t.join() for t in ths]
    return voice, sl


def run_reference(args, wl, group):
    """--impl reference: the reference's own CPU implementation on the host cores, rank 0 only."""
    if group.rank != 0:
        return
    # inputs from the stand-alone generator: nothing of the product is loaded into this process (built by
    # __graft_entry__.build(); if it is missing, the product's own vp_synth_host -- same definitions -- generates them)
    vp = None
    if not os.path.exists(os.path.join(ROOT, "tools", "_build", "libvp_inputgen.so")):
        import vocoderproject_b200 as vp
    fs, B = wl["fs"], wl["B"]
    n = int(fs * wl["seconds"]) // B * B
    cores = host_cores()
    S = max(1, min(wl["streams"], args.ref_streams or 2 * cores))
    voice, sl = gen_host_inputs(vp, fs, 0, S, n, cores)
    kind = "reference"
    for _ in range(args.warmup):
        cpu_run("reference", fs, B, voice, sl, wl["params"], cores)
    t = 0.0
    for _ in range(args.steps):
        sec, kind = cpu_run("reference", fs, B, voice, sl, wl["params"], cores)
        t += sec
    audio = S * n / fs * args.steps
    val = audio / t
    line = {"impl": "reference", "metric": "audio-sec/sec (streams x RT)", "value": val, "unit": "audio-s/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl["desc"], "sample_rate": fs, "block": B, "seconds_per_stream": n / fs,
                       "params": wl["params"] or "defaults"},
            "cpu_baseline": {"value": val, "unit": "audio-s/s", "cores": cores, "kind": kind,
                             "sample": "%d streams x %.1f s of the workload per step, one plug-in instance per stream, %d host threads"
                                       % (S, n / fs, cores)},
            "e2e": {"value": val, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_engine(args, wl, group):
    os.environ["VP_STAGE_TIMING"] = "1"      # CUDA events between the engine's kernels (per-kernel durations)
    os.environ["VP_KEEP_DECISIONS"] = "1"    # per-frame decisions of every stream stay on the device: the parity check below reads a spread of them
    import vocoderproject_b200 as vp
    fs, B = wl["fs"], wl["B"]
    n = int(fs * wl["seconds"]) // B * B
    nBlocks = n // B
    S = args.streams or wl["streams"]          # per GPU (weak scaling)
    first = group.rank * S                      # global stream index of this shard
    dev = group.local_rank
    prm = vp.default_params(**wl["params"])
    eng = vp.Engine(fs, B, S, nBlocks, params=prm, device=dev)
    sz = eng.sizes
    nb = S * n * 4
    dv, dl, do = eng.device_alloc(nb), eng.device_alloc(nb), eng.device_alloc(nb)
    eng.synth_device(0, first, S, n, n, dv, dl, None)
    peaks_fp = eng.measure_peaks()
    sampler = ClockSampler(dev)

    # ---- device-resident: W warm-up + K timed steps, barrier + sync on both sides
    # every step = prepareToPlay + the whole batch: reset() rewinds the streams (consecutive calls would continue them)
    for _ in range(args.warmup):
        eng.reset()
        eng.process_device(nBlocks, dv, dl, None, do, None, n, sync=False)
    eng.sync()
    l0 = eng.stats()["kernel_launches"]
    eng.timing_reset(accumulate=True)
    group.barrier()
    t0 = time.time()
    eng.timer_record(0)
    for _ in range(args.steps):
        eng.reset()
        eng.process_device(nBlocks, dv, dl, None, do, None, n, sync=False)
    eng.timer_record(1)
    eng.sync()
    t1 = time.time()
    group.barrier()
    dev_s = eng.timer_elapsed_ms(0, 1) * 1e-3
    launches = eng.stats()["kernel_launches"] - l0
    tot_ms, stage_ms = eng.last_timing()
    stage_cnt = eng.last_timing_counts()
    eng.timing_reset(accumulate=False)
    clocks = sampler.window(t0, t1)
    audio_rank = S * n / fs * args.steps
    value, t_max, audio_total = vp.shard.aggregate_throughput(group, audio_rank, dev_s)
    dump = dump_outputs(eng, do, S, n, group, args.dump_outputs) if args.dump_outputs else None

    # ---- parity at the benchmarked size: a spread of streams of the LAST timed step, full length, against the reference
    # on the host cores (oracle/_ref, else the C port). Test infrastructure used as the checker only.
    parity, picks, dev_rows = None, [], {}
    if not args.no_parity:
        parity, picks, dev_rows = parity_check(vp, eng, args, wl, S, n, dv, dl, do, group)

    # ---- end to end through the host-buffer C-ABI call (pinned host memory, H2D + D2H inside)
    e2e = None
    cpu_from_pinned = True
    if not args.no_e2e:
        # pinned host memory for the whole batch: 3 arrays per rank; fall back to fewer streams if the box is short
        Se = S
        try:
            avail = [int(l.split()[1]) * 1024 for l in open("/proc/meminfo") if l.startswith("MemAvailable")][0]
            budget = 0.6 * avail / max(group.world, 1)
            while Se > 32 and 3.0 * Se * n * 4 > budget:
                Se //= 2
        except Exception:
            pass
        numa = numa_bind(dev)
        hv, hl, ho = vp.PinnedArray(Se, n), vp.PinnedArray(Se, n), vp.PinnedArray(Se, n)
        eng.d2h(hv.array, dv)
        eng.d2h(hl.array, dl)
        for p in (dv, dl, do):
            eng.device_free(p)
        dv = dl = do = None
        if Se != S:  # a smaller engine for the end-to-end leg (same per-stream workload)
            eng.close()
            eng = vp.Engine(fs, B, Se, nBlocks, params=prm, device=dev)
        audio_rank_e = Se * n / fs * args.steps
        nb_e = Se * n * 4
        we = max(1, min(args.warmup, 2))
        for _ in range(we):
            eng.reset()
            eng.process_host_ptrs(nBlocks, hv.ptr, hl.ptr, None, ho.ptr, None, n)
        group.barrier()
        te0 = time.time()
        for _ in range(args.steps):
            eng.reset()
            eng.process_host_ptrs(nBlocks, hv.ptr, hl.ptr, None, ho.ptr, None, n)  # returns with outputs in host memory
        te = time.time() - te0
        group.barrier()
        e_val, e_t, _ = vp.shard.aggregate_throughput(group, audio_rank_e, te)
        if parity is not None:  # the host path must return what the device-resident path left in HBM, bit for bit
            same = all(np.array_equal(ho.array[s_], dev_rows[s_]) for s_ in picks if s_ < Se)
            parity["e2e_rows_equal_device_rows"] = bool(group.min(1.0 if same else 0.0) > 0.5)
        e2e_checksum = float(np.abs(ho.array[:, ::4097]).sum())
        # the host link's rates on this box, now (fallback: the committed probe log for this GPU count)
        link = live_link_probe(group, dev, hv.ptr, ho.ptr, min(1 << 30, nb_e)) or link_ceiling(group.world)
        link_info = None
        if link:
            lb = link_bound(link, 2.0 * nb_e * group.world, 1.0 * nb_e * group.world)
            link_info = {"h2d_alone_gbs": link["h2d"], "d2h_alone_gbs": link["d2h"], "duplex_total_gbs": link["duplex"], "lower_bound_ms": 1e3 * lb,
                         "achieved_gbs": 3.0 * nb_e * group.world / (e_t / args.steps) / 1e9,
                         "model": "max(h2d bytes / h2d-alone rate, d2h bytes / d2h-alone rate, all bytes / both-directions total rate)",
                         "source": (os.path.relpath(link["file"], ROOT) + ": pinned 1-D copies, %d GPU(s) copying at once" % group.world) if link.get("file")
                                   else "measured in this run (tools/link_probe.cu's method): pinned 1-D copies of %.2f GiB, %d GPU(s) copying at once" % (link["live_gib"], group.world)}
        e2e = {"value": e_val, "unit": "audio-s/s", "h2d_bytes_per_step": 2 * nb_e * group.world, "d2h_bytes_per_step": nb_e * group.world,
               "streams_per_gpu": Se, "numa": numa, "link": link_info,
               "link_frac": (link_info["lower_bound_ms"] / (1e3 * e_t / args.steps)) if link_info else None,
               "ms_per_step": 1e3 * e_t / args.steps, "timer": "host wall clock around vp_engine_process_host, max over ranks",
               "note": "voice + side-chain ch0 uploaded (the path reads ch0 only, VocoderProcess.cpp:211,218); one output channel "
                       "returned (L == R while gainSynth <= -59 dB)", "checksum": e2e_checksum}
        if not args.no_pcm16:
            # the same batch as 16-bit PCM across the link (vp_engine_process_host_pcm16): the float rows are quantised in
            # place into the first half of their own pinned buffers (row s of the int16 view ends before row s of the floats)
            qv = np.frombuffer((C.c_int16 * (Se * n)).from_address(hv.ptr), dtype=np.int16).reshape(Se, n)
            ql = np.frombuffer((C.c_int16 * (Se * n)).from_address(hl.ptr), dtype=np.int16).reshape(Se, n)
            def quantise(pair):  # rows in increasing order per array: row s of the int16 view never reaches an unread float row
                q_, f_ = pair
                for s_ in range(Se):
                    q_[s_] = np.clip(np.rint(f_[s_] * np.float32(32768.0)), -32768, 32767).astype(np.int16)
            ths = [threading.Thread(target=quantise, args=(pr,)) for pr in ((qv, hv.array), (ql, hl.array))]
            [t.start() for t in ths]
            [t.join() for t in ths]
            ksteps = args.steps
            eng.reset()
            eng.process_host_pcm16_ptrs(nBlocks, hv.ptr, hl.ptr, None, ho.ptr, None, n)
            group.barrier()
            tq0 = time.time()
            for _ in range(ksteps):
                eng.reset()
                eng.process_host_pcm16_ptrs(nBlocks, hv.ptr, hl.ptr, None, ho.ptr, None, n)
            tq = time.time() - tq0
            group.barrier()
            q_val, q_t, _ = vp.shard.aggregate_throughput(group, Se * n / fs * ksteps, tq)
            qo = np.frombuffer((C.c_int16 * (Se * n)).from_address(ho.ptr), dtype=np.int16).reshape(Se, n)
            e2e["pcm16"] = {"value": q_val, "unit": "audio-s/s", "steps": ksteps, "ms_per_step": 1e3 * q_t / ksteps,
                            "h2d_bytes_per_step": nb_e * group.world, "d2h_bytes_per_step": nb_e // 2 * group.world,
                            "link_frac": (1e3 * link_bound(link, 1.0 * nb_e * group.world, 0.5 * nb_e * group.world) / (1e3 * q_t / ksteps)) if link else None,
                            "workload": "same batch, 16-bit PCM host arrays through vp_engine_process_host_pcm16 (int16 <-> float on the device, "
                                        "bit-identical to csrc/vp_wav.hpp's host conversion); an extension for PCM sources, not a format of the reference's processBlock",
                            "checksum": int(np.abs(qo[:, ::4097].astype(np.int64)).sum())}
            cpu_from_pinned = False
        else:
            cpu_from_pinned = True
    sampler.stop()

    # ---- CPU baseline on rank 0 at N = 1: bounded sample of the same workload
    cpu = None
    if group.world == 1 and not args.no_cpu:
        cores = host_cores()
        Sc = max(1, min(S if e2e is None else Se, args.cpu_streams or 8 * cores))
        secs_cpu = min(n / fs, 20.0)
        ncpu = int(fs * secs_cpu) // B * B
        if e2e is not None and cpu_from_pinned:
            cv, cl = np.ascontiguousarray(hv.array[:Sc, :ncpu]), np.ascontiguousarray(hl.array[:Sc, :ncpu])
        elif e2e is not None:  # the pinned float inputs were quantised in place for the PCM16 leg: generate the sample again
            cv, cl = gen_host_inputs(vp, fs, first, Sc, ncpu, cores)
        else:
            cv = np.zeros((Sc, n), np.float32); cl = np.zeros((Sc, n), np.float32)
            for s in range(Sc):  # row copies of the device inputs
                eng.lib.vp_memcpy_d2h(eng.h, cv[s].ctypes.data, C.c_void_p(dv + s * n * 4), n * 4)
                eng.lib.vp_memcpy_d2h(eng.h, cl[s].ctypes.data, C.c_void_p(dl + s * n * 4), n * 4)
            cv, cl = np.ascontiguousarray(cv[:, :ncpu]), np.ascontiguousarray(cl[:, :ncpu])
        sec, kind = cpu_run("reference", fs, B, cv, cl, wl["params"], cores)
        cpu = {"value": Sc * ncpu / fs / sec, "unit": "audio-s/s", "cores": cores, "kind": kind,
               "sample": "%d streams x %.1f s of the workload (%.1f s wall), one plug-in instance per stream, %d host threads, "
                         "-O3 build of the reference's own C++" % (Sc, ncpu / fs, sec, cores)}

    if group.rank == 0:
        sm = slot_model(sz, prm)
        peaks, peaks_src = measured_peaks()
        p32 = peaks_fp["fp32_fma_per_s"]
        samples_rank = S * n * args.steps
        chain_slots = (sm["voc_per_sample"] if prm.vocBool else 0.0) + (sm["pitch_per_sample"] if prm.pitchBool else 0.0)
        # dominant kernel: the stage with the largest share of the device time
        # (the pitch-mark chain runs on a side stream UNDER the vocoder kernels: its time overlaps theirs and is not a share of the step)
        kname = max((k for k in stage_ms if k != "marks"), key=lambda k: stage_ms[k])
        kms, kcnt = stage_ms[kname], max(stage_cnt.get(kname, 1), 1)
        frames_v = S * ((n + sz["hopV"] - 1) // sz["hopV"]) * args.steps
        frames_p = S * ((n + sz["hopP"] - 1) // sz["hopP"]) * args.steps
        kslots = {"yin_fp32": sm["pitch"]["yin"] * frames_p,
                  "voc_autocorr": (sm["voc"]["window"] + sm["voc"]["autocorr_voice"] + sm["voc"]["autocorr_synth"]) * frames_v,
                  "voc_levinson": (sm["voc"]["levinson"] + sm["voc"]["fir_voice"] + sm["voc"]["fir_synth"]) * frames_v,
                  "voc_synth": (sm["voc"]["gain"] + sm["voc"]["iir"] + sm["voc"]["ola"] + sm["voc"]["fir_synth"]) * frames_v,
                  "pitch_lpc": (sm["pitch"]["autocorr"] + sm["pitch"]["levinson"]) * frames_p,
                  "pitch_psola": (sm["pitch"]["residual_fir"] + sm["pitch"]["psola"]) * frames_p,
                  "pitch_iir": (sm["pitch"]["iir"] + sm["pitch"]["ola"]) * frames_p}.get(kname, 0.0)
        # the same stage counted as the FP64 multiply-adds its algorithm needs (these kernels run on the FP64 pipe)
        wl_, ov_, os_, op_ = sz["wlenV"], prm.lpcVoice, prm.lpcSynth, prm.lpcPitch
        kdfma = {"voc_synth": (ov_ + os_ + 1) * wl_ * frames_v,
                 "voc_autocorr": (sum(wl_ - m for m in range(ov_ + 1)) + sum(wl_ - m for m in range(os_ + 1))) * frames_v,
                 "pitch_psola": (sz["tauMax"] + sz["frameLenP"] + 3 * sz["chunk"]) * (op_ + 1) * frames_p,
                 "pitch_iir": op_ * sz["frameLenP"] * frames_p}.get(kname)
        ach = 2.0 * kslots / (kms * 1e-3) / 1e12 if kms > 0 else 0.0
        peak = 2.0 * p32 / 1e12
        io_bytes = 12.0 * samples_rank  # voice + synth ch0 in, one channel out (float32)
        # DRAM bytes of that kernel from the committed ncu --set full capture (per sample there), scaled to one launch here
        traffic, traffic_note = None, None
        mcap = mix_capture(args.workload)
        if mcap and kname in mcap["stages"]:
            traffic = mcap["stages"][kname]["dram_bytes_per_sample"] * samples_rank / kcnt
            traffic_note = "dram__bytes_read.sum + dram__bytes_write.sum of the %s kernels in %s, per sample x samples of one launch" % (kname, mcap["source"])
        try:
            if traffic is not None:
                raise LookupError
            import glob
            with open(sorted(glob.glob(os.path.join(ROOT, "profiles", "ncu_traffic_*.json")))[-1]) as f:  # newest capture
                tj = json.load(f)
            if kname in tj["stages"] and wl["fs"] == 48000.0 and not wl["params"]:
                traffic = tj["stages"][kname]["dram_bytes_per_sample"] * samples_rank / kcnt
                traffic_note = "dram__bytes_read.sum + dram__bytes_write.sum of %s in %s, per sample x samples of one launch" % (
                    tj["stages"][kname]["kernel"], tj["source"])
        except Exception:
            pass
        roofline = {"bound": "fp32", "kernel": kname, "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak if peak else None,
                    "traffic": traffic, "traffic_note": traffic_note, "kernel_ms_per_launch": kms / kcnt, "kernel_launches_timed": kcnt,
                    "kernel_share_of_step": kms / tot_ms if tot_ms else None,
                    "peak_source": "vp_measure_peaks FP32 FMA issue-rate microbenchmark on this GPU in this run (2 flop per lane-op); "
                                   "MEASURED_PEAKS.json (%s) has no FP32 CUDA-core figure" % peaks_src,
                    "note": "algorithmic FP32 lane-ops of the minimal direct form (SURVEY App. C.5), 1 lane-op counted as 2 flop on both sides",
                    "fp64": (None if kdfma is None else {"achieved_tdfma_per_s": kdfma / (kms * 1e-3) / 1e12, "peak_tdfma_per_s": peaks_fp["fp64_fma_per_s"] / 1e12,
                                                         "frac": kdfma / (kms * 1e-3) / peaks_fp["fp64_fma_per_s"],
                                                         "note": "this kernel is FP64-pipe bound: algorithmic DFMAs / event time vs the measured DFMA issue rate"}),
                    "chain": {"slots_per_sample": chain_slots, "achieved_tflops": 2.0 * chain_slots * samples_rank / dev_s / 1e12,
                              "frac": chain_slots * samples_rank / dev_s / p32 if p32 else None,
                              "note": "direct-form op count of SURVEY App. C.5 (the contract number); roofline.mix is the same step against "
                                      "the instructions the kernels execute"},
                    "mix": mix_roofline(args.workload, float(S) * n, 1e3 * dev_s / args.steps, peaks_fp, clocks.get("sm_max_mhz")),
                    "hbm": {"achieved_gbs": io_bytes / dev_s / 1e9, "peak_gbs": peaks.get("hbm_gbs"), "peak_source": peaks_src,
                            "frac": io_bytes / dev_s / 1e9 / peaks.get("hbm_gbs", 1.0), "algorithmic_bytes_per_sample": 12},
                    "fp64_fma_per_s": peaks_fp["fp64_fma_per_s"], "fp32_fma_per_s": p32,
                    "fp32_fma_2op_per_s": peaks_fp.get("fp32_fma_2op_per_s"), "fp64_fma_2op_per_s": peaks_fp.get("fp64_fma_2op_per_s"),
                    "stage_ms": {k: round(v, 3) for k, v in stage_ms.items() if v > 0}, "stage_launches": {k: v for k, v in stage_cnt.items() if v}}
        line = {"metric": "audio-sec/sec (streams x RT)", "value": value, "unit": "audio-s/s", "n_gpus": group.world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1e3 * t_max / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
                "config": {"workload": wl["desc"], "sample_rate": fs, "block": B, "streams_per_gpu": S, "streams_total": S * group.world,
                           "seconds_per_stream": n / fs, "params": wl["params"] or "defaults", "parallelism": "streams sharded x%d, no collective" % group.world,
                           "l2": "inputs (%.1f GB per GPU) far larger than the 126 MB L2; no flush needed" % (2 * nb / 1e9),
                           "timer": "CUDA events on the engine's stream around the K steps, max over ranks"},
                "x_realtime_per_gpu": value / group.world, "clocks": clocks, "gpu_launches": int(launches) * group.world,
                "roofline": roofline}
        if e2e is not None:
            line["e2e"] = e2e
        if parity is not None:
            line["parity"] = parity
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if dump is not None:
            line["dump_outputs"] = dump
    eng.close()
    if group.world == 1 and not args.no_sub and not args.streams and args.workload == "chain48":
        # the other BASELINE configurations, driver-observed: chain @ 44.1 kHz is the north_star target line
        line["other_workloads"] = {}
        for name in ("chain44", "voc44", "pitch44"):
            try:
                line["other_workloads"][name] = run_sub(vp, args, name, group, peaks_fp, clocks.get("sm_max_mhz"))
            except Exception as ex:
                line["other_workloads"][name] = {"error": str(ex)}
    if group.rank == 0:
        if group.world == 1 and not args.no_stream and not args.streams:
            try:
                line["streaming"] = run_streaming(args, group)
            except Exception as ex:  # the throughput line must not depend on the latency sub-test
                line["streaming"] = {"error": str(ex)}
        print(json.dumps(line), flush=True)


def parity_check(vp, eng, args, wl, S, n, dv, dl, do, group):
    """>= 16 streams spread over this rank's [0, S) -- incl. the first and last stream of every pass -- for their full
    length: inputs and outputs copied back from HBM, the reference run on the same inputs on the host cores, audio SNR /
    max |err| and every pitch decision compared (tests/common.py). Returns (parity dict aggregated over ranks, picks, rows)."""
    from common import MAXABS_MAX, SNR_MIN_DB, compare_decisions, maxabs, oracle_decisions, reference_runs, snr_db
    fs, B = wl["fs"], wl["B"]
    Sc = eng.info()["streams_per_pass"]
    picks = set()
    for p0 in range(0, S, Sc):
        picks |= {p0, min(p0 + Sc, S) - 1}
    want = max(args.parity_streams, len(picks))
    for x in np.linspace(0, S - 1, want):
        if len(picks) >= want:
            break
        picks.add(int(round(x)))
    picks = sorted(picks)
    ins, outs = [], {}
    for s_ in picks:
        v, l, o_ = np.zeros(n, np.float32), np.zeros(n, np.float32), np.zeros(n, np.float32)
        for arr, base in ((v, dv), (l, dl), (o_, do)):
            eng._check(eng.lib.vp_memcpy_d2h(eng.h, arr.ctypes.data, C.c_void_p(base + s_ * n * 4), n * 4))
        ins.append((fs, B, v, l, None, wl["params"]))
        outs[s_] = o_
    t0 = time.time()
    refs, kind = reference_runs(ins)
    cpu_s = time.time() - t0
    worst_snr, worst_abs, tot, chk, flg, exc, bad = 1e9, 0.0, 0, 0, 0, 0, 0
    first = None
    prm_pitch = wl["params"].get("pitchBool", 1)
    for s_, r in zip(picks, refs):
        worst_snr = min(worst_snr, snr_db(r["outL"], outs[s_]))
        worst_abs = max(worst_abs, maxabs(r["outL"], outs[s_]))
        if prm_pitch:
            dec = compare_decisions(vp, oracle_decisions(r["pitch"]), eng.pitch_frames(s_))
            tot += dec.n; chk += dec.checked; flg += dec.flagged; exc += dec.excused; bad += dec.bad
            if dec.bad and first is None:
                first = "stream %d: %s" % (s_, dec.first)
    st = eng.stats()
    res = {"streams": int(group.sum(len(picks))), "streams_per_rank": len(picks), "seconds": n / fs, "reference": kind,
           "worst_snr_db": group.min(worst_snr), "worst_maxabs": group.max(worst_abs),
           "frames": int(group.sum(tot)), "frames_compared": int(group.sum(chk)), "frames_flagged": int(group.sum(flg)),
           "frames_excused": int(group.sum(exc)), "mismatches": int(group.sum(bad)),
           "recheck_list_overflow": False,  # vp_engine_sync turns an overflow into an error (and the list holds every frame)
           "yin_rechecked_frac": (st["yin_rechecked"] / float(S * ((n + eng.sizes["hopP"] - 1) // eng.sizes["hopP"]))) if prm_pitch else 0.0,
           "tolerance": {"snr_db_min": SNR_MIN_DB, "maxabs_max": MAXABS_MAX, "decisions": "bit-exact, checked >= 98 % of frames"},
           "streams_checked_rank0": picks, "cpu_seconds": cpu_s}
    ok = (res["worst_snr_db"] >= SNR_MIN_DB and res["worst_maxabs"] <= MAXABS_MAX and res["mismatches"] == 0 and
          res["frames_compared"] >= 0.98 * res["frames"])
    res["ok"] = bool(ok)
    if first:
        res["first_mismatch"] = first
    if not ok:
        if group.rank == 0:
            print(json.dumps({"parity_failed": res}), file=sys.stderr, flush=True)
        raise SystemExit("bench.py: parity check at the benchmarked size FAILED: %r" % ({k: res[k] for k in ("worst_snr_db", "worst_maxabs", "mismatches", "frames", "frames_compared")},))
    return res, picks, outs


def run_streaming(args, group):
    """BASELINE configs[4]: 4096 concurrent streams, block 128 @ 44.1 kHz, one CUDA-graph launch per block; latency of
    vp_engine_stream_block = enqueue -> the block's outputs visible in pinned host memory."""
    import vocoderproject_b200 as vp
    fs, B, S = 44100.0, 128, args.streams or 4096
    nb = args.stream_blocks
    eng = vp.Engine(fs, B, S, 1, params=vp.default_params(), device=group.local_rank)
    hv, hs, ho = eng.stream_buffers()
    # a few seconds of distinct input per stream would not fit the point of the test: cycle 64 pre-generated blocks
    nsrc = 64
    src_v, src_s, _ = vp.synth_host(fs, min(S, 64), nsrc * B, flavour=0, first_stream=0)
    reps = (S + src_v.shape[0] - 1) // src_v.shape[0]
    src_v = np.tile(src_v, (reps, 1))[:S]
    src_s = np.tile(src_s, (reps, 1))[:S]
    lat = []
    for b in range(nb + 32):
        k = b % nsrc
        hv[:] = src_v[:, k * B:(k + 1) * B]
        hs[:] = src_s[:, k * B:(k + 1) * B]
        t0 = time.perf_counter()
        eng.stream_block()
        t1 = time.perf_counter()
        if b >= 32:  # graphs of all block phases captured during the first 32 blocks
            lat.append((t1 - t0) * 1e3)
    st = eng.stream_stats()
    eng.close()
    lat = np.array(lat)
    res = {"workload": "streaming: %d concurrent streams, block %d @ 44.1 kHz, full chain, CUDA graph per block" % (S, B),
           "blocks_timed": int(len(lat)), "block_period_ms": 1e3 * B / fs, "p50_ms": float(np.percentile(lat, 50)),
           "p99_ms": float(np.percentile(lat, 99)), "max_ms": float(lat.max()), "mean_ms": float(lat.mean()),
           "realtime_margin_p99": float(1e3 * B / fs / np.percentile(lat, 99)), "graph_captures": st["graph_captures"],
           "timer": "host perf_counter around vp_engine_stream_block (pinned H2D + graph + pinned D2H + sync)"}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--workload", default="chain48", choices=sorted(WORKLOADS))
    ap.add_argument("--streams", type=int, default=0, help="streams per GPU (default: the workload's)")
    ap.add_argument("--seconds", type=float, default=0.0, help="seconds per stream (default: the workload's)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-pcm16", action="store_true", help="skip the 16-bit PCM end-to-end leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle comparison at the benchmarked size")
    ap.add_argument("--parity-streams", type=int, default=16, help="streams per rank compared with the reference")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-sub", action="store_true", help="skip the short runs of the other BASELINE configurations")
    ap.add_argument("--cpu-streams", type=int, default=0)
    ap.add_argument("--ref-streams", type=int, default=0)
    ap.add_argument("--stream-blocks", type=int, default=1500, help="blocks timed by the streaming latency test")
    ap.add_argument("--no-stream", action="store_true", help="skip the streaming (p99 block latency) sub-test")
    ap.add_argument("--stream-only", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed, seeded sample (at most 64 MB) of the output of the last timed step as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.impl != "engine" or args.stream_only):
        ap.error("--dump-outputs writes the outputs of the engine's batch run: not with --impl reference or --stream-only")
    if args.warmup < 3 and args.impl == "engine":
        print("note: --warmup < 3 breaks the timing rules; use it for smoke runs only", file=sys.stderr)
    wl = dict(WORKLOADS[args.workload])
    if args.seconds:
        wl["seconds"] = args.seconds
        wl["desc"] += " [--seconds %g]" % args.seconds
    if args.streams:
        wl["desc"] += " [--streams %d]" % args.streams
    from vocoderproject_b200.shard import Group, dist_env
    rank, _, world = dist_env()
    if args.impl == "reference":
        if rank != 0:
            return 0  # rank 0 alone runs the CPU reference
        class Solo:
            rank, local_rank, world = 0, 0, 1
        run_reference(args, wl, Solo())
        return 0
    if world != args.gpus and world > 1:
        print("warning: WORLD_SIZE=%d but --gpus %d; using WORLD_SIZE" % (world, args.gpus), file=sys.stderr)
    if world == 1 and args.gpus > 1:
        # convenience: relaunch under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus), "--master-addr", "127.0.0.1",
               "--master-port", "29533", os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    group = Group()
    try:
        if args.stream_only:
            if group.rank == 0:
                print(json.dumps({"metric": "p99 block latency", "unit": "ms", "higher_is_better": False, **run_streaming(args, group)}), flush=True)
            return 0
        run_engine(args, wl, group)
    finally:
        group.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
