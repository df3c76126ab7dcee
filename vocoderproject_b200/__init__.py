"""vocoderproject_b200 -- Python host mirror of the B200 batch engine's C ABI
(include/vp_engine.h). The product is the CUDA shared library
vocoderproject_b200/lib/libvp_engine.so; this module only binds it with ctypes
(numpy for host buffers). There is no CPU fallback: if the library is missing
or no CUDA device is usable, every compute call raises."""
import ctypes as C
import os

import numpy as np

from . import shard  # noqa: F401  (stream sharding over GPUs; no data-path collective)

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libvp_engine.so")

VP_OK, VP_E_ARG, VP_E_STATE, VP_E_CUDA, VP_E_NOMEM, VP_E_RANGE = 0, -1, -2, -3, -4, -5
VP_MAX_MARKS = 24
VP_MODE_PARITY, VP_MODE_DEFINED = 0, 1
VP_WINDOW_SINE, VP_WINDOW_HANN = 0, 1
VP_NSTAGES = 16
VP_SNAPSHOT_VERSION, VP_SNAPSHOT_HEADER_BYTES, VP_SNAPSHOT_RECORD_BYTES = 1, 352, 144
PF_GATED, PF_VOICED, PF_HAS_MARKS = 1, 2, 4
PF_NEAR_GATE, PF_NEAR_YIN, PF_UB, PF_YIN_RECHECKED = 16, 32, 64, 128

# every symbol include/vp_engine.h declares (checked by tests/test_abi.py)
ABI_SYMBOLS = [
    "vp_default_params", "vp_sizes_for", "vp_device_count", "vp_engine_create", "vp_engine_destroy",
    "vp_last_error", "vp_engine_prepare", "vp_engine_set_params", "vp_engine_get_sizes",
    "vp_engine_process_device", "vp_engine_process_host", "vp_engine_sync", "vp_engine_get_pitch_frames",
    "vp_engine_get_voc_frames", "vp_engine_get_stats", "vp_engine_last_timing", "vp_stage_name",
    "vp_host_alloc", "vp_host_free", "vp_device_alloc", "vp_device_free", "vp_memcpy_h2d", "vp_memcpy_d2h",
    "vp_synth_host", "vp_synth_device", "vp_measure_peaks", "vp_engine_timing_reset", "vp_engine_timer_record",
    "vp_engine_timer_elapsed_ms", "vp_engine_last_timing_counts", "vp_measure_peaks2", "vp_engine_reset", "vp_engine_stream_buffers", "vp_engine_stream_block",
    "vp_engine_stream_stats", "vp_engine_get_info", "vp_engine_reserve_orders", "vp_grid_plan", "vp_engine_set_mode", "vp_engine_process_host_pcm16", "vp_engine_set_window",
    "vp_engine_set_stream_params", "vp_engine_get_stream_params", "vp_engine_reset_streams", "vp_engine_schedule_stream_params",
    "vp_engine_set_stream_orders", "vp_engine_get_stream_orders", "vp_engine_schedule_stream_orders",
    "vp_engine_reserve_pitch_order", "vp_engine_set_stream_pitch_orders", "vp_engine_get_stream_pitch_orders",
    "vp_engine_snapshot_size", "vp_engine_save_streams", "vp_engine_load_streams",
]


class Params(C.Structure):
    _fields_ = [("gainPitch", C.c_float), ("gainVoice", C.c_float), ("gainSynth", C.c_float),
                ("gainVoc", C.c_float), ("lpcVoice", C.c_int), ("lpcPitch", C.c_int), ("lpcSynth", C.c_int),
                ("keyPitch", C.c_int), ("pitchBool", C.c_int), ("vocBool", C.c_int)]


class StreamParams(C.Structure):
    """vp_stream_params: the per-instance part of Params (key and gains of one stream)."""
    _fields_ = [("gainPitch", C.c_float), ("gainVoice", C.c_float), ("gainSynth", C.c_float), ("gainVoc", C.c_float),
                ("keyPitch", C.c_int)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


STREAM_PARAM_FIELDS = tuple(k for k, _ in StreamParams._fields_)


class StreamEvent(C.Structure):
    """vp_stream_event: stream `stream` takes p from absolute block `block` on (blocks since prepare / reset). 40 bytes."""
    _fields_ = [("stream", C.c_int), ("reserved", C.c_int), ("block", C.c_longlong), ("p", StreamParams), ("pad", C.c_int)]


class StreamOrders(C.Structure):
    """vp_stream_orders: the vocoder's two LPC orders of one stream. 8 bytes."""
    _fields_ = [("lpcVoice", C.c_int), ("lpcSynth", C.c_int)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


STREAM_ORDER_FIELDS = tuple(k for k, _ in StreamOrders._fields_)


class StreamOrderEvent(C.Structure):
    """vp_stream_order_event: stream `stream` takes the orders o from absolute block `block` on. 24 bytes."""
    _fields_ = [("stream", C.c_int), ("reserved", C.c_int), ("block", C.c_longlong), ("o", StreamOrders)]


def stream_params(**kw):
    """StreamParams with the plug-in's defaults (gains 0 / -60 / -60 / 0 dB, chromatic key), overridden by kw."""
    p = StreamParams(0.0, -60.0, -60.0, 0.0, 12)
    for k, v in kw.items():
        if k not in STREAM_PARAM_FIELDS:
            raise KeyError(k)
        setattr(p, k, v)
    return p


class Sizes(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("hopV", "wlenV", "hopP", "frameLenP", "chunk", "tauMin", "tauMax",
                                       "latency", "keep", "inSize", "outSize", "anCap", "nFreq")]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class PitchFrame(C.Structure):
    _fields_ = [("flags", C.c_uint32), ("period", C.c_int32), ("periodPsola", C.c_int32),
                ("periodNew", C.c_int32), ("note", C.c_int32), ("nAn", C.c_int32), ("nSt", C.c_int32),
                ("anStale", C.c_int32), ("nAnOv", C.c_int32), ("prevAnLast", C.c_int32), ("anMarks", C.c_int32 * VP_MAX_MARKS),
                ("stMarks", C.c_int32 * VP_MAX_MARKS), ("beta", C.c_double)]


class CallPlan(C.Structure):
    _fields_ = [("firstBlock", C.c_longlong), ("offV", C.c_int), ("nFramesV", C.c_int), ("carriedV", C.c_int),
                ("rowOrderV", C.c_int), ("rowOrderS", C.c_int), ("offP", C.c_int), ("nFramesP", C.c_int),
                ("vocMix", C.c_int), ("pitchMix", C.c_int), ("rowsOrphaned", C.c_int), ("orphansLive", C.c_int),
                ("carryPosP", C.c_int * 2), ("carryChunksP", C.c_int * 2)]


class EngineError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("vp_engine error %d: %s" % (code, msg))
        self.code = code


_lib = None


def load_library(path=None):
    """Loads libvp_engine.so (building nothing: see vocoderproject_b200.build)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise EngineError(VP_E_STATE, "%s not built; run `python -m vocoderproject_b200.build` (needs nvcc). "
                                      "There is no CPU fallback." % path)
    lib = C.CDLL(path)
    vp, fp, i, sz, dbl = C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_double
    sig = {
        "vp_default_params": (None, [C.POINTER(Params)]),
        "vp_sizes_for": (i, [dbl, i, i, C.POINTER(Sizes)]),
        "vp_device_count": (i, []),
        "vp_engine_create": (i, [C.POINTER(vp), i]),
        "vp_engine_destroy": (None, [vp]),
        "vp_last_error": (C.c_char_p, [vp]),
        "vp_engine_prepare": (i, [vp, dbl, i, i, i, sz]),
        "vp_engine_set_params": (i, [vp, C.POINTER(Params)]),
        "vp_engine_set_stream_params": (i, [vp, i, i, C.POINTER(StreamParams)]),
        "vp_engine_get_stream_params": (i, [vp, i, i, C.POINTER(StreamParams)]),
        "vp_engine_get_sizes": (i, [vp, C.POINTER(Sizes)]),
        "vp_engine_get_info": (i, [vp, C.POINTER(i), C.POINTER(i), C.POINTER(sz)]),
        "vp_engine_reserve_orders": (i, [vp, i, i]),
        "vp_engine_set_mode": (i, [vp, i]),
        "vp_engine_set_window": (i, [vp, i]),
        "vp_grid_plan": (i, [dbl, i, i, C.POINTER(i), C.POINTER(Params), C.POINTER(CallPlan)]),
        "vp_engine_process_device": (i, [vp, i, fp, fp, fp, fp, fp, sz]),
        "vp_engine_process_host": (i, [vp, i, fp, fp, fp, fp, fp, sz]),
        "vp_engine_process_host_pcm16": (i, [vp, i, fp, fp, fp, fp, fp, sz]),
        "vp_engine_sync": (i, [vp]),
        "vp_engine_get_pitch_frames": (i, [vp, i, C.POINTER(PitchFrame), i, C.POINTER(i)]),
        "vp_engine_get_voc_frames": (i, [vp, i, i, C.POINTER(i), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
        "vp_engine_get_stats": (i, [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
        "vp_engine_last_timing": (i, [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
        "vp_stage_name": (C.c_char_p, [i]),
        "vp_host_alloc": (i, [C.POINTER(vp), sz]),
        "vp_host_free": (None, [vp]),
        "vp_device_alloc": (i, [vp, C.POINTER(vp), sz]),
        "vp_device_free": (None, [vp, vp]),
        "vp_memcpy_h2d": (i, [vp, vp, vp, sz]),
        "vp_memcpy_d2h": (i, [vp, vp, vp, sz]),
        "vp_synth_host": (i, [dbl, i, i, i, sz, sz, fp, fp, fp]),
        "vp_synth_device": (i, [vp, dbl, i, i, i, sz, sz, fp, fp, fp]),
        "vp_measure_peaks": (i, [vp, C.POINTER(dbl), C.POINTER(dbl)]),
        "vp_engine_timing_reset": (i, [vp, i]),
        "vp_engine_reset": (i, [vp]),
        "vp_engine_reset_streams": (i, [vp, C.POINTER(i), i]),
        "vp_engine_schedule_stream_params": (i, [vp, C.POINTER(StreamEvent), i]),
        "vp_engine_set_stream_orders": (i, [vp, i, i, C.POINTER(StreamOrders)]),
        "vp_engine_get_stream_orders": (i, [vp, i, i, C.POINTER(StreamOrders)]),
        "vp_engine_schedule_stream_orders": (i, [vp, C.POINTER(StreamOrderEvent), i]),
        "vp_engine_reserve_pitch_order": (i, [vp, i]),
        "vp_engine_set_stream_pitch_orders": (i, [vp, i, i, C.POINTER(i)]),
        "vp_engine_get_stream_pitch_orders": (i, [vp, i, i, C.POINTER(i), C.POINTER(i)]),
        "vp_engine_snapshot_size": (i, [vp, i, C.POINTER(sz)]),
        "vp_engine_save_streams": (i, [vp, C.POINTER(i), i, C.c_void_p, sz]),
        "vp_engine_load_streams": (i, [vp, C.POINTER(i), i, C.c_char_p, sz]),
        "vp_engine_stream_buffers": (i, [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]),
        "vp_engine_stream_block": (i, [vp]),
        "vp_engine_stream_stats": (i, [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
        "vp_measure_peaks2": (i, [vp, C.POINTER(dbl), C.POINTER(dbl)]),
        "vp_engine_last_timing_counts": (i, [vp, C.POINTER(i)]),
        "vp_engine_timer_record": (i, [vp, i]),
        "vp_engine_timer_elapsed_ms": (i, [vp, i, i, C.POINTER(C.c_float)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def default_params(**kw):
    p = Params()
    load_library().vp_default_params(C.byref(p))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise KeyError(k)
        setattr(p, k, v)
    return p


def sizes_for(sample_rate, block, key=12):
    s = Sizes()
    rc = load_library().vp_sizes_for(float(sample_rate), int(block), int(key), C.byref(s))
    if rc != VP_OK:
        raise EngineError(rc, "vp_sizes_for(%r, %r, %r)" % (sample_rate, block, key))
    return s.as_dict()


def grid_plan(sample_rate, block, calls):
    """calls: [(nBlocks, Params), ...] -> list of CallPlan (host-only: the frame grids those process calls produce)."""
    n = len(calls)
    nb = (C.c_int * n)(*[int(c[0]) for c in calls])
    ps = (Params * n)()
    for k, (_, q) in enumerate(calls):
        C.memmove(C.byref(ps[k]), C.byref(q), C.sizeof(Params))
    out = (CallPlan * n)()
    rc = load_library().vp_grid_plan(float(sample_rate), int(block), n, nb, ps, out)
    if rc != VP_OK:
        raise EngineError(rc, "vp_grid_plan")
    return list(out)


def synth_host(sample_rate, n_streams, n_samples, flavour=0, first_stream=0, want_right=True):
    """Synthetic voice / side-chain inputs generated on the host (float32 [S][n])."""
    lib = load_library()
    voice = np.zeros((n_streams, n_samples), np.float32)
    sl = np.zeros_like(voice)
    sr = np.zeros_like(voice) if want_right else None
    rc = lib.vp_synth_host(float(sample_rate), flavour, first_stream, n_streams, n_samples, n_samples,
                           voice.ctypes.data, sl.ctypes.data, sr.ctypes.data if sr is not None else None)
    if rc != VP_OK:
        raise EngineError(rc, "vp_synth_host")
    return voice, sl, sr


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return a


class PinnedArray:
    """float32 [rows][cols] in CUDA pinned host memory (vp_host_alloc)."""

    def __init__(self, rows, cols):
        self._lib = load_library()
        p = C.c_void_p()
        nbytes = int(rows) * int(cols) * 4
        rc = self._lib.vp_host_alloc(C.byref(p), nbytes)
        if rc != VP_OK:
            raise EngineError(rc, "vp_host_alloc(%d bytes)" % nbytes)
        self.ptr = p.value
        buf = (C.c_float * (int(rows) * int(cols))).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=np.float32).reshape(rows, cols)

    def free(self):
        if self.ptr:
            self.array = None
            self._lib.vp_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Engine:
    """N independent plug-in instances on one GPU.

    Mirrors the reference's call order (PluginProcessor.cpp:144-234):
    Engine(...) ~ construct + set parameters + prepareToPlay(sampleRate, samplesPerBlock);
    process(...) ~ nBlocks consecutive processBlock calls per stream."""

    def __init__(self, sample_rate, block, n_streams, max_blocks, params=None, device=0, workspace_bytes=0, reserve_orders=None,
                 window=VP_WINDOW_SINE, reserve_pitch_order=None):
        self.lib = load_library()
        self.h = C.c_void_p()
        rc = self.lib.vp_engine_create(C.byref(self.h), int(device))
        if rc != VP_OK:
            self.h = None
            raise EngineError(rc, "vp_engine_create failed (no usable CUDA device %d; there is no CPU fallback)" % device)
        self.sample_rate, self.block, self.n_streams, self.max_blocks = float(sample_rate), int(block), int(n_streams), int(max_blocks)
        self.params = params or default_params()
        if window != VP_WINDOW_SINE:
            self._check(self.lib.vp_engine_set_window(self.h, int(window)))
        if reserve_orders:  # (maxLpcVoice, maxLpcSynth) that set_params may be given while the streams run
            self._check(self.lib.vp_engine_reserve_orders(self.h, int(reserve_orders[0]), int(reserve_orders[1])))
        if reserve_pitch_order:  # largest lpcPitch that set_stream_pitch_orders may be given
            self._check(self.lib.vp_engine_reserve_pitch_order(self.h, int(reserve_pitch_order)))
        self._check(self.lib.vp_engine_set_params(self.h, C.byref(self.params)))
        self._check(self.lib.vp_engine_prepare(self.h, self.sample_rate, self.block, self.n_streams, self.max_blocks,
                                               int(workspace_bytes)))
        s = Sizes()
        self._check(self.lib.vp_engine_get_sizes(self.h, C.byref(s)))
        self.sizes = s.as_dict()

    def _check(self, rc):
        if rc != VP_OK:
            msg = self.lib.vp_last_error(self.h)
            raise EngineError(rc, msg.decode() if msg else "")

    def close(self):
        if getattr(self, "h", None):
            self.lib.vp_engine_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self):
        """Layout chosen at prepare: streams per pass, carried history length, workspace bytes."""
        a, b, c = C.c_int(0), C.c_int(0), C.c_size_t(0)
        self._check(self.lib.vp_engine_get_info(self.h, C.byref(a), C.byref(b), C.byref(c)))
        return {"streams_per_pass": a.value, "history_samples": b.value, "workspace_bytes": c.value}

    def reset(self):
        """prepareToPlay again: forget every stream's history; the next process call starts at block 0."""
        self._check(self.lib.vp_engine_reset(self.h))

    def reset_streams(self, streams):
        """Hand the listed streams to new instances: from the next process call on, each continues as a stream that has
        heard only silence since prepare (its key and gains are kept, its pending scheduled changes are dropped). The other
        streams are not touched."""
        streams = [int(s) for s in streams]
        arr = (C.c_int * max(len(streams), 1))(*streams)
        self._check(self.lib.vp_engine_reset_streams(self.h, arr, len(streams)))

    # ---- per-stream state snapshots: move a running stream to another slot or engine, checkpoint a render ----
    def snapshot_size(self, count):
        """Bytes of a snapshot of `count` streams (header + count records) for this engine as prepared."""
        n = C.c_size_t(0)
        self._check(self.lib.vp_engine_snapshot_size(self.h, int(count), C.byref(n)))
        return n.value

    def save_streams(self, streams):
        """The state the listed streams start their next process call with, as an opaque, self-checking blob (bytes).
        Waits for every call already issued; changes nothing in the engine."""
        streams = [int(s) for s in streams]
        arr = (C.c_int * max(len(streams), 1))(*streams)
        n = self.snapshot_size(len(streams))
        buf = C.create_string_buffer(n)
        self._check(self.lib.vp_engine_save_streams(self.h, arr, len(streams), buf, n))
        return buf.raw

    def load_streams(self, streams, blob):
        """Record i of blob (save_streams of this or a compatible engine) becomes the state of slot streams[i]: same layout
        key, same grid phase, or this engine has processed no block since prepare / reset (it then adopts the blob's grids).
        Validated before anything is issued; on an error nothing changes."""
        streams = [int(s) for s in streams]
        arr = (C.c_int * max(len(streams), 1))(*streams)
        blob = bytes(blob)
        self._check(self.lib.vp_engine_load_streams(self.h, arr, len(streams), blob, len(blob)))

    # ---- low-latency streaming: one host block per call through pinned buffers and a CUDA graph per block phase ----
    def stream_buffers(self):
        """(voice, synthL, outL): numpy views [S][B] of the engine's pinned host buffers."""
        pv, ps, po = C.c_void_p(), C.c_void_p(), C.c_void_p()
        self._check(self.lib.vp_engine_stream_buffers(self.h, C.byref(pv), C.byref(ps), C.byref(po)))
        shape = (self.n_streams, self.block)

        def view(p):
            buf = (C.c_float * (shape[0] * shape[1])).from_address(p.value)
            return np.frombuffer(buf, dtype=np.float32).reshape(shape)
        return view(pv), view(ps), view(po)

    def stream_block(self):
        self._check(self.lib.vp_engine_stream_block(self.h))

    def stream_stats(self):
        a, b = C.c_uint64(0), C.c_uint64(0)
        self._check(self.lib.vp_engine_stream_stats(self.h, C.byref(a), C.byref(b)))
        return {"graph_launches": a.value, "graph_captures": b.value}

    def set_mode(self, mode):
        """VP_MODE_PARITY (the reference as it runs) or VP_MODE_DEFINED (bounds-correct at its undefined-behaviour sites)."""
        self._check(self.lib.vp_engine_set_mode(self.h, int(mode)))

    def set_params(self, params):
        """Engine-wide parameters; the key, the gains and the vocoder orders go to every stream (replacing per-stream values)."""
        self._check(self.lib.vp_engine_set_params(self.h, C.byref(params)))
        self.params = params

    def set_stream_params(self, first, items):
        """Key and gains of streams first .. first + len(items) - 1; items are StreamParams or dicts (missing fields of a
        dict keep the stream's current value). Takes effect with the next process call."""
        items = list(items)
        cur = self.stream_params(first, len(items)) if any(isinstance(it, dict) for it in items) else None
        arr = (StreamParams * max(len(items), 1))()
        for k, it in enumerate(items):
            if isinstance(it, StreamParams):
                C.memmove(C.byref(arr[k]), C.byref(it), C.sizeof(StreamParams))
            else:
                for f in STREAM_PARAM_FIELDS:
                    setattr(arr[k], f, it[f] if f in it else cur[k][f])
                for f in it:
                    if f not in STREAM_PARAM_FIELDS:
                        raise KeyError(f)
        self._check(self.lib.vp_engine_set_stream_params(self.h, int(first), len(items), arr))

    def schedule_stream_params(self, events):
        """Block-accurate automation: events = [(stream, block, values), ...]; stream `stream` takes the values from absolute
        block `block` on (blocks since prepare / reset; not one already processed), where the reference reads each of them --
        also inside one multi-block process call. values is a StreamParams or a dict; the missing fields of a dict are the
        stream's values just before that block as far as this call can tell: its current values, updated by the earlier
        events of the same list for that stream at blocks up to that one (events queued by earlier calls are not seen).
        On an error nothing is queued."""
        events = list(events)
        cur = None
        if any(not isinstance(v, StreamParams) for _, _, v in events):
            cur = self.stream_params()
        # for dicts: the mirror of each stream's values, in block order (a stable sort keeps list order within a block)
        order = sorted(range(len(events)), key=lambda k: (int(events[k][1]), k))
        last = {}
        arr = (StreamEvent * max(len(events), 1))()
        for k in order:
            s, b, v = events[k]
            s, b = int(s), int(b)
            e = arr[k]
            e.stream, e.block, e.reserved, e.pad = s, b, 0, 0
            if isinstance(v, StreamParams):
                C.memmove(C.byref(e.p), C.byref(v), C.sizeof(StreamParams))
                vals = v.as_dict()
            else:
                for f in v:
                    if f not in STREAM_PARAM_FIELDS:
                        raise KeyError(f)
                base = last.get(s) or (cur[s] if 0 <= s < len(cur) else dict(stream_params().as_dict()))
                vals = dict(base)
                vals.update(v)
                for f in STREAM_PARAM_FIELDS:
                    setattr(e.p, f, vals[f])
            last[s] = vals
        self._check(self.lib.vp_engine_schedule_stream_params(self.h, arr, len(events)))

    def stream_params(self, first=0, count=None):
        """[dict] of the key and gains of streams first .. first + count - 1 (default: to the last stream)."""
        if count is None:
            count = self.n_streams - int(first)
        arr = (StreamParams * max(int(count), 1))()
        self._check(self.lib.vp_engine_get_stream_params(self.h, int(first), int(count), arr))
        return [arr[k].as_dict() for k in range(int(count))]

    def set_stream_orders(self, first, items):
        """Vocoder orders (lpcVoice, lpcSynth) of streams first .. first + len(items) - 1; items are StreamOrders, dicts
        (missing fields keep the stream's current value) or (lpcVoice, lpcSynth) pairs. Takes effect from the next block on,
        at each vocoder frame start."""
        items = list(items)
        cur = self.stream_orders(first, len(items)) if any(isinstance(it, dict) for it in items) else None
        arr = (StreamOrders * max(len(items), 1))()
        for k, it in enumerate(items):
            if isinstance(it, StreamOrders):
                C.memmove(C.byref(arr[k]), C.byref(it), C.sizeof(StreamOrders))
            elif isinstance(it, dict):
                for f in it:
                    if f not in STREAM_ORDER_FIELDS:
                        raise KeyError(f)
                for f in STREAM_ORDER_FIELDS:
                    setattr(arr[k], f, int(it[f] if f in it else cur[k][f]))
            else:
                arr[k].lpcVoice, arr[k].lpcSynth = int(it[0]), int(it[1])
        self._check(self.lib.vp_engine_set_stream_orders(self.h, int(first), len(items), arr))

    def stream_orders(self, first=0, count=None):
        """[dict] of the vocoder orders of streams first .. first + count - 1 (default: to the last stream)."""
        if count is None:
            count = self.n_streams - int(first)
        arr = (StreamOrders * max(int(count), 1))()
        self._check(self.lib.vp_engine_get_stream_orders(self.h, int(first), int(count), arr))
        return [arr[k].as_dict() for k in range(int(count))]

    def set_stream_pitch_orders(self, first, values):
        """lpcPitch of streams first .. first + len(values) - 1: the order each starts with. In force from the next process
        call for a stream that has processed no block since its last start (prepare, reset, or a pending reset_streams of
        it); any other stream keeps its order until its next start."""
        values = [int(v) for v in values]
        arr = (C.c_int * max(len(values), 1))(*values)
        self._check(self.lib.vp_engine_set_stream_pitch_orders(self.h, int(first), len(values), arr))

    def stream_pitch_orders(self, first=0, count=None):
        """(in_force, next): lists of the lpcPitch each of streams first .. first + count - 1 runs its next block at, and the
        one it takes at its next start (default count: to the last stream)."""
        if count is None:
            count = self.n_streams - int(first)
        a = (C.c_int * max(int(count), 1))()
        b = (C.c_int * max(int(count), 1))()
        self._check(self.lib.vp_engine_get_stream_pitch_orders(self.h, int(first), int(count), a, b))
        return [a[k] for k in range(int(count))], [b[k] for k in range(int(count))]

    def schedule_stream_orders(self, events):
        """Block-accurate order automation: events = [(stream, block, orders), ...] with the rules of
        schedule_stream_params; orders is a StreamOrders, a (lpcVoice, lpcSynth) pair or a dict whose missing fields are
        the stream's orders just before that block as far as this call can tell. On an error nothing is queued."""
        events = list(events)
        cur = self.stream_orders() if any(isinstance(v, dict) for _, _, v in events) else None
        order = sorted(range(len(events)), key=lambda k: (int(events[k][1]), k))
        last = {}
        arr = (StreamOrderEvent * max(len(events), 1))()
        for k in order:
            s, b, v = events[k]
            s, b = int(s), int(b)
            e = arr[k]
            e.stream, e.block, e.reserved = s, b, 0
            if isinstance(v, StreamOrders):
                vals = v.as_dict()
            elif isinstance(v, dict):
                for f in v:
                    if f not in STREAM_ORDER_FIELDS:
                        raise KeyError(f)
                base = last.get(s) or (cur[s] if 0 <= s < len(cur) else {"lpcVoice": 40, "lpcSynth": 5})
                vals = dict(base)
                vals.update(v)
            else:
                vals = {"lpcVoice": int(v[0]), "lpcSynth": int(v[1])}
            e.o.lpcVoice, e.o.lpcSynth = int(vals["lpcVoice"]), int(vals["lpcSynth"])
            last[s] = vals
        self._check(self.lib.vp_engine_schedule_stream_orders(self.h, arr, len(events)))

    # ---- host-buffer API (what a plug-in host calls) ----
    def process(self, voice, synthL, synthR=None, want_right=True):
        """voice/synthL/synthR: float32 [S][n] host arrays; returns (outL, outR) [S][nBlocks*B]."""
        voice = np.ascontiguousarray(voice, np.float32)
        synthL = np.ascontiguousarray(synthL, np.float32)
        if synthR is not None:
            synthR = np.ascontiguousarray(synthR, np.float32)
        S, n = voice.shape
        assert S == self.n_streams and synthL.shape == voice.shape
        nBlocks = n // self.block
        outL = np.zeros((S, n), np.float32)
        outR = np.zeros((S, n), np.float32) if want_right else None
        self._check(self.lib.vp_engine_process_host(self.h, nBlocks, _ptr(voice), _ptr(synthL), _ptr(synthR),
                                                    _ptr(outL), _ptr(outR), n))
        m = nBlocks * self.block
        return outL[:, :m], (outR[:, :m] if outR is not None else None)

    def process_pcm16(self, voice, synthL, synthR=None, want_right=True):
        """int16 [S][n] host arrays in and out (vp_engine_process_host_pcm16): 16-bit PCM across the host link."""
        voice = np.ascontiguousarray(voice, np.int16)
        synthL = np.ascontiguousarray(synthL, np.int16)
        if synthR is not None:
            synthR = np.ascontiguousarray(synthR, np.int16)
        S, n = voice.shape
        nBlocks = n // self.block
        outL = np.zeros((S, n), np.int16)
        outR = np.zeros((S, n), np.int16) if want_right else None
        self._check(self.lib.vp_engine_process_host_pcm16(self.h, nBlocks, _ptr(voice), _ptr(synthL), _ptr(synthR), _ptr(outL), _ptr(outR), n))
        m = nBlocks * self.block
        return outL[:, :m], (outR[:, :m] if outR is not None else None)

    def process_host_pcm16_ptrs(self, n_blocks, voice, synthL, synthR, outL, outR, stride):
        self._check(self.lib.vp_engine_process_host_pcm16(self.h, int(n_blocks), _ptr(voice), _ptr(synthL), _ptr(synthR), _ptr(outL), _ptr(outR), int(stride)))

    def process_host_ptrs(self, n_blocks, voice, synthL, synthR, outL, outR, stride):
        self._check(self.lib.vp_engine_process_host(self.h, int(n_blocks), _ptr(voice), _ptr(synthL), _ptr(synthR),
                                                    _ptr(outL), _ptr(outR), int(stride)))

    # ---- device-buffer API ----
    def device_alloc(self, nbytes):
        p = C.c_void_p()
        self._check(self.lib.vp_device_alloc(self.h, C.byref(p), int(nbytes)))
        return p.value

    def device_free(self, p):
        self.lib.vp_device_free(self.h, p)

    def h2d(self, dst, src_array):
        self._check(self.lib.vp_memcpy_h2d(self.h, dst, src_array.ctypes.data, src_array.nbytes))

    def d2h(self, dst_array, src):
        self._check(self.lib.vp_memcpy_d2h(self.h, dst_array.ctypes.data, src, dst_array.nbytes))

    def process_device(self, n_blocks, voice, synthL, synthR, outL, outR, stride, sync=True):
        self._check(self.lib.vp_engine_process_device(self.h, int(n_blocks), voice, synthL, synthR, outL, outR, int(stride)))
        if sync:
            self.sync()

    def sync(self):
        self._check(self.lib.vp_engine_sync(self.h))

    def synth_device(self, flavour, first_stream, n_streams, n_samples, stride, voice, synthL, synthR):
        self._check(self.lib.vp_synth_device(self.h, self.sample_rate, int(flavour), int(first_stream), int(n_streams),
                                             int(n_samples), int(stride), voice, synthL, synthR))

    # ---- decisions / stats ----
    def pitch_frames(self, stream):
        n = C.c_int(0)
        self._check(self.lib.vp_engine_get_pitch_frames(self.h, int(stream), None, 0, C.byref(n)))
        if n.value == 0:
            return []
        buf = (PitchFrame * n.value)()
        self._check(self.lib.vp_engine_get_pitch_frames(self.h, int(stream), buf, n.value, C.byref(n)))
        return list(buf)

    def voc_frames(self, stream):
        n = C.c_int(0)
        self._check(self.lib.vp_engine_get_voc_frames(self.h, int(stream), 0, C.byref(n), None, None, None, None))
        m = n.value
        gated = np.zeros(m, np.uint8)
        ev, es, g = np.zeros(m), np.zeros(m), np.zeros(m)
        if m:
            self._check(self.lib.vp_engine_get_voc_frames(self.h, int(stream), m, C.byref(n), gated.ctypes.data,
                                                          ev.ctypes.data, es.ctypes.data, g.ctypes.data))
        return {"gated": gated, "EeVoice": ev, "EeSynth": es, "g": g}

    def stats(self):
        a, b, c = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        self._check(self.lib.vp_engine_get_stats(self.h, C.byref(a), C.byref(b), C.byref(c)))
        return {"kernel_launches": a.value, "yin_rechecked": b.value, "yin_frames": c.value}

    def last_timing(self):
        tot = C.c_float(0)
        st = (C.c_float * VP_NSTAGES)()
        self._check(self.lib.vp_engine_last_timing(self.h, C.byref(tot), st))
        return tot.value, {self.lib.vp_stage_name(i).decode(): st[i] for i in range(VP_NSTAGES)}

    def last_timing_counts(self):
        cnt = (C.c_int * VP_NSTAGES)()
        self._check(self.lib.vp_engine_last_timing_counts(self.h, cnt))
        return {self.lib.vp_stage_name(i).decode(): cnt[i] for i in range(VP_NSTAGES)}

    def timing_reset(self, accumulate=False):
        self._check(self.lib.vp_engine_timing_reset(self.h, 1 if accumulate else 0))

    def timer_record(self, slot):
        self._check(self.lib.vp_engine_timer_record(self.h, int(slot)))

    def timer_elapsed_ms(self, a, b):
        ms = C.c_float(0)
        self._check(self.lib.vp_engine_timer_elapsed_ms(self.h, int(a), int(b), C.byref(ms)))
        return ms.value

    def measure_peaks(self):
        a, b = C.c_double(0), C.c_double(0)
        self._check(self.lib.vp_measure_peaks(self.h, C.byref(a), C.byref(b)))
        c2, d2 = C.c_double(0), C.c_double(0)
        self._check(self.lib.vp_measure_peaks2(self.h, C.byref(c2), C.byref(d2)))
        return {"fp32_fma_per_s": a.value, "fp64_fma_per_s": b.value, "fp32_fma_2op_per_s": c2.value, "fp64_fma_2op_per_s": d2.value}
