"""Generate tests/golden/pins_ref.json: the results of the UNMODIFIED reference headers (oracle/_ref, built over minieigen by
`make -C oracle ref` where the reference tree is present) on the inputs of tests/util.py:pin_cases, which
tests/test_oracle_cpu.py's test_pin_* hold the restatement to, bit for bit.

    python tests/golden/make_pins.py

Arrays are stored as SHA-256 digests of their bytes (tests/util.py:fingerprint): a failing pin says which field differs.
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import pyoracle as po  # noqa: E402
from util import PIN_GROUPS, fingerprint, pin_cases  # noqa: E402


def main():
    ref = po.Oracle("ref")
    groups = {g: {name: fingerprint(run(ref)) for name, run in pin_cases(g)} for g in PIN_GROUPS}
    out = os.path.join(HERE, "pins_ref.json")
    with open(out, "w") as fh:
        json.dump(dict(generator="tests/golden/make_pins.py", source="oracle/_ref (unmodified reference headers @ ebef584 over oracle/minieigen)",
                       groups=groups), fh, indent=0, sort_keys=True)
        fh.write("\n")
    print("wrote", out, sum(len(v) for v in groups.values()), "cases,", os.path.getsize(out) // 1024, "KiB")


if __name__ == "__main__":
    main()
