"""Golden-fixture cases: seeded synthetic inputs (vp_synth_host / SURVEY App. E
generator) x plug-in parameter sets. tests/golden/make_golden.py runs the
REFERENCE (oracle/_ref, the reference's C++ compiled in place) on them in the
authoring container and commits the outputs; the tests replay them through the
CPU oracle (not gpu) and through the CUDA engine (gpu)."""

# name -> dict(fs, B, seconds, input=("synth", flavour, firstStream) | ("kat",), params={...})
CASES = {
    # SURVEY.md section 8(d) config 1 flavour: chain, C major, 44.1 kHz, B = 1024
    "chain44_cmaj": dict(fs=44100.0, B=1024, seconds=2.0, input=("synth", 0, 0), params=dict(keyPitch=3)),
    # config 4 flavour: chain, chromatic, 48 kHz
    "chain48_chrom": dict(fs=48000.0, B=1024, seconds=2.0, input=("synth", 0, 1), params=dict()),
    # config 2 flavour: vocoder only, on the clean (-80 dBFS noise) voice = the FP64 stress case
    "voc44_clean": dict(fs=44100.0, B=1024, seconds=2.0, input=("synth", 1, 2), params=dict(pitchBool=0)),
    # config 3 flavour: pitch corrector only, chromatic
    "pitch44_chrom": dict(fs=44100.0, B=1024, seconds=2.0, input=("synth", 0, 3), params=dict(vocBool=0)),
    # config 5 flavour: streaming block size
    "chain44_b128": dict(fs=44100.0, B=128, seconds=2.0, input=("synth", 0, 4), params=dict()),
    # ragged block size + dry voice / dry synth mix (stereo differs) + non-default gains
    "chain44_b1000_mix": dict(fs=44100.0, B=1000, seconds=2.0, input=("synth", 0, 5),
                              params=dict(gainVoice=-6.0, gainSynth=-12.0, gainVoc=-3.0, gainPitch=2.0, keyPitch=7)),
    # non-default LPC orders
    "chain44_orders": dict(fs=44100.0, B=512, seconds=1.5, input=("synth", 0, 6),
                           params=dict(lpcVoice=24, lpcSynth=8, lpcPitch=20)),
    # parameter automation between blocks (what a DAW does to the plug-in's atomics): gains and key change mid-stream
    "chain44_automation": dict(fs=44100.0, B=512, seconds=3.0, input=("synth", 0, 7),
                               params=dict(keyPitch=3, gainVoice=-20.0, gainSynth=-30.0),
                               schedule=[(40, dict(gainVoc=-6.0, gainPitch=3.0)), (97, dict(keyPitch=12)),
                                         (150, dict(gainVoice=-60.0, gainSynth=-10.0, keyPitch=7)),
                                         (201, dict(gainVoc=2.0, gainPitch=-4.0, keyPitch=0))]),
    # every parameter automated, incl. the LPC orders (per vocoder frame, VocoderProcess.cpp:193-194) and the two enables (per
    # block, PluginProcessor.cpp:214-221; pitchBool off = PitchProcess::silence()); lpcPitch mid-stream is ignored (read in
    # prepare only). The schedule of tests/test_oracle.py::test_oracle_automation_bit_exact_vs_reference_build.
    "chain44_toggles": dict(fs=44100.0, B=256, seconds=2.5, input=("synth", 0, 77), params=dict(keyPitch=5, gainSynth=-25.0),
                            reserve=(64, 9),
                            schedule=[(30, dict(lpcVoice=20, lpcSynth=9)), (77, dict(gainVoc=-4.0, keyPitch=12, gainVoice=-12.0)),
                                      (120, dict(pitchBool=0)), (160, dict(pitchBool=1, lpcVoice=64, keyPitch=1)), (200, dict(vocBool=0)),
                                      (260, dict(vocBool=1, gainPitch=-7.0, lpcSynth=3)), (330, dict(lpcPitch=9))]),
    # 48 kHz, block 128: hop 139 and chunk 278 are larger than the block, so a skipped block makes the frame grids slip
    # against the blocks, frames in flight outlive short off-stretches (orphaned vocoder frames, cut pitch frames)
    "chain48_b128_toggles": dict(fs=48000.0, B=128, seconds=2.0, input=("synth", 0, 8), params=dict(keyPitch=3),
                                 reserve=(48, 8),
                                 schedule=[(100, dict(vocBool=0)), (101, dict(vocBool=1)), (140, dict(vocBool=0)), (143, dict(vocBool=1, lpcVoice=24)),
                                           (200, dict(pitchBool=0)), (201, dict(pitchBool=1)), (260, dict(pitchBool=0, vocBool=0)),
                                           (263, dict(pitchBool=1)), (266, dict(vocBool=1, lpcVoice=48, lpcSynth=8)),
                                           (400, dict(pitchBool=0)), (407, dict(pitchBool=1, lpcVoice=40, lpcSynth=5)),
                                           (500, dict(vocBool=0, gainVoice=-10.0)), (520, dict(vocBool=1)), (600, dict(vocBool=0)), (601, dict(vocBool=1))]),
    # 48 kHz, block 1024: whole blocks of vocoder / pitch corrector switched off; and the dry side-chain switched ON mid-stream
    # (gainSynth off -> on: the first `latency` samples it adds come from the right channel's ring of the blocks before,
    # which is filled whatever gainSynth is, MyBuffer.cpp:69-92) and off / on again
    "chain48_b1024_toggles": dict(fs=48000.0, B=1024, seconds=2.5, input=("synth", 0, 9), params=dict(),
                                  schedule=[(20, dict(vocBool=0)), (22, dict(vocBool=1)), (30, dict(gainSynth=-12.0)), (40, dict(pitchBool=0)),
                                            (41, dict(pitchBool=1)), (60, dict(vocBool=0, pitchBool=0)), (63, dict(vocBool=1, pitchBool=1)),
                                            (70, dict(gainSynth=-60.0)), (80, dict(gainSynth=-6.0)), (90, dict(pitchBool=0))]),
    # the "hann" window type of VocoderProcess::setWindows (VocoderProcess.cpp:116-124: rectangular analysis, Hann synthesis),
    # which prepareToPlay never selects: the harness calls the reference's own setWindows("hann") after prepareToPlay
    "chain44_hann": dict(fs=44100.0, B=1024, seconds=2.0, input=("synth", 0, 10), params=dict(keyPitch=3), window="hann"),
    # leading silence -> gates (vocoder + pitch) then voiced onset; KAT-style inputs delayed by 0.5 s
    "gate_onset": dict(fs=44100.0, B=1024, seconds=2.0, input=("kat_delayed", 22050), params=dict(keyPitch=3)),
}

# SURVEY.md App. E known-answer table (produced by the survey's own throw-away harness,
# independent of oracle/ref_harness.cpp): 4 s, fs 44100, B 1024, keyPitch 3.
KAT = {
    "chain": dict(params=dict(keyPitch=3), first_nonzero=1024, sum=-245.458814, sum_abs=53330.001634, rms=0.37169441,
                  max_abs=0.89971805, samples={5000: 0.454756349, 50000: 0.025890775, 150000: -0.26012823},
                  crc="c1d66746"),
    "voc": dict(params=dict(keyPitch=3, pitchBool=0), first_nonzero=1024, sum=-1.436721, sum_abs=43512.132665,
                rms=0.27328791, max_abs=0.47363758, samples={5000: 0.25661841, 50000: -0.168966845, 150000: 0.0170496777},
                crc="36fe865c"),
    "pitch": dict(params=dict(keyPitch=3, vocBool=0), first_nonzero=1537, sum=-244.022094, sum_abs=38165.470135,
                  rms=0.25202407, max_abs=0.46377969, samples={5000: 0.198137909, 50000: 0.194857627, 150000: -0.2771779},
                  crc="f9b1e16c"),
}
# frame : startSample : anMarks : stMarks (SURVEY.md App. E)
KAT_MARKS = {
    2: (512, [151, 374, 593, 815], [151, 376, 601, 826]),
    3: (256, [47, 269, 488, 710, 931], [58, 283, 508, 733, 958]),
    4: (0, [163, 383, 604, 827], [190, 415, 640, 865]),
    5: (768, [59, 278, 500, 720, 941], [97, 322, 547, 772, 997]),
    6: (512, [173, 394, 615, 836], [4, 229, 454, 679, 904]),
    7: (256, [68, 290, 510, 731, 954], [136, 361, 586, 811]),
    8: (0, [186, 407, 627, 848], [43, 268, 493, 718, 943]),
    9: (768, [80, 300, 521, 742, 963], [175, 400, 625, 850]),
}
KAT_PERIOD, KAT_NOTE, KAT_BETA, KAT_PERIODNEW = 221, 6, 0.9822107863034768, 225

# (fs, B, keyPitch, flavour) of tests/test_oracle.py::test_oracle_bit_exact_vs_reference_build: block sizes and rates the
# golden fixtures above do not cover. Their pins are in tests/golden/reference_build_pins.json.
REF_BUILD_CASES = [(44100.0, 64, 3, 0), (48000.0, 1000, 12, 1), (44100.0, 128, 0, 0)]


def ref_build_inputs(vp, fs, B, flavour):
    """(voice, synthL, synthR) float32 [n] of a REF_BUILD_CASES entry: 1.5 s of whole blocks."""
    n = int(fs * 1.5) // B * B
    v, l, r = vp.synth_host(fs, 1, n, flavour=flavour, first_stream=40 + B)
    return v[0], l[0], r[0]


def ref_build_key(fs, B, key, flavour):
    return "fs=%g,B=%d,key=%d,flavour=%d" % (fs, B, key, flavour)


def case_schedule(case):
    """[(block, cumulative parameter dict), ...] of a case ('schedule' entries override what is in force so far)."""
    cur = dict(case["params"])
    out = []
    for b, d in case.get("schedule", []):
        cur = dict(cur, **d)
        out.append((b, dict(cur)))
    return out


def case_inputs(vp, case):
    """(voice, synthL, synthR) float32 [n] for a case; n = whole blocks."""
    import numpy as np
    from common import kat_inputs
    fs, B = case["fs"], case["B"]
    n = int(fs * case["seconds"]) // B * B
    kind = case["input"][0]
    if kind == "synth":
        _, flavour, first = case["input"]
        v, l, r = vp.synth_host(fs, 1, n, flavour=flavour, first_stream=first)
        return v[0], l[0], r[0]
    if kind == "kat_delayed":
        d = case["input"][1]
        v, s = kat_inputs(int(fs), int(np.ceil(case["seconds"])))
        vo = np.zeros(n, np.float32)
        so = np.zeros(n, np.float32)
        vo[d:] = v[:n - d]
        so[d:] = s[:n - d]
        return vo, so, so.copy()
    raise KeyError(kind)
