"""Writes tests/golden/reference_build_pins.json: what tests/test_oracle.py::test_oracle_bit_exact_vs_reference_build
compares the oracle with, for the cases of tests/cases.py REF_BUILD_CASES, so that the test runs where the reference's
sources are absent.

    python tests/golden/make_reference_pins.py

It runs the reference build (oracle/_ref/libvpref_strict.so) when that is built, else the C restatement
(oracle/libvp_oracle.so), and records which in "source". The committed file was written by the C restatement: the
reference's sources were not at hand, and on these three cases the restatement is bit-exact with the reference build
(DESIGN.md section 2; the same test compares the two whenever oracle/_ref is built)."""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
sys.path[:0] = [ROOT, TESTS]

import vocoderproject_b200 as vp  # noqa: E402  (host-side synthetic input generator only)
import oraclebind  # noqa: E402
import refbind  # noqa: E402
from cases import REF_BUILD_CASES, ref_build_inputs, ref_build_key  # noqa: E402
from common import reference_pin  # noqa: E402


def main():
    use_ref = refbind.available("strict")
    pins = {"source": "oracle/_ref/libvpref_strict.so (the reference build)" if use_ref else
            "oracle/libvp_oracle.so (the C restatement, bit-exact with the reference build on these cases)"}
    for fs, B, key, flavour in REF_BUILD_CASES:
        v, l, r = ref_build_inputs(vp, fs, B, flavour)
        prm = refbind.default_params(keyPitch=key)
        run = refbind.run if use_ref else oraclebind.run
        pins[ref_build_key(fs, B, key, flavour)] = reference_pin(run(fs, B, v, l, synthR=r, params=prm, log=True))
    with open(os.path.join(HERE, "reference_build_pins.json"), "w") as f:  # one line per pitch frame
        text = json.dumps(pins, indent=1, sort_keys=True)
        for name, pin in pins.items():
            if name != "source":
                for row in pin["decisions"]:
                    text = text.replace(json.dumps(row, indent=1, sort_keys=True).replace("\n", "\n   "),
                                        json.dumps(row, sort_keys=True), 1)
        assert json.loads(text) == pins
        f.write(text + "\n")


if __name__ == "__main__":
    main()
