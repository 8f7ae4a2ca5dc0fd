"""Writes reference_outputs.json: what the reference's own code returns on the seeded inputs of
tests/test_reference_pin.py and tests/test_gpu_vs_reference_build.py (their `reference_outputs(R)`).

Needs oracle/_ref/libvlcal_ref.so, the reference's sources of the path compiled against the stand-in headers of
oracle/ref_standin (`make -C oracle ref REF=<reference source tree>`).  The tests compare the oracle and the CUDA path
with the stored file, so they run without the reference tree or its build.
    python tests/golden/make_reference_outputs.py
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

from oracle import reference as R  # noqa: E402
import test_gpu_vs_reference_build  # noqa: E402
import test_reference_pin  # noqa: E402
import util  # noqa: E402


def main():
    if R.build() is None:
        raise SystemExit(f"{R.LIB_PATH} is missing: build it with `make -C oracle ref REF=<reference source tree>`")
    out = {**test_reference_pin.reference_outputs(R), **test_gpu_vs_reference_build.reference_outputs(R)}
    with open(util.REFERENCE_OUTPUTS, "w") as f:
        json.dump(util.plain(out), f, indent=0, sort_keys=True)
        f.write("\n")
    print("written", util.REFERENCE_OUTPUTS)


if __name__ == "__main__":
    main()
