"""Writes tests/golden/reference_api.json: the API surface of the reference operator that this project keeps.

    python tools/record_reference_api.py REFERENCE_CHECKOUT      # regenerate (review the diff before committing!)

Recorded from the reference's Go sources: every JSON field name of its API types, every string constant of its API
package, every command-line flag of its options, and the SHA-256 of its example manifest.  tests/test_reference_parity.py
checks this project against the recording, so the check needs no reference checkout.
"""
import glob
import hashlib
import json
import os
import re
import sys

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "reference_api.json")


def record(ref: str) -> dict:
    api = [f for f in sorted(glob.glob(os.path.join(ref, "pkg/apis/aitrainingjob/v1/*.go"))) if "zz_generated" not in f]
    if not api:
        raise SystemExit(f"{ref}: no pkg/apis/aitrainingjob/v1/*.go")
    tags, consts = set(), set()
    for f in api:
        src = open(f).read()
        tags |= set(re.findall(r'json:"([^",]+)', src))
        consts |= set(re.findall(r'\b\w+(?:\s+\w+)?\s*=\s*"([^"]+)"', src))
    flags = set(re.findall(r'fs\.\w+\([^"]*"([\w-]+)"', open(os.path.join(ref, "cmd/app/options/options.go")).read()))
    example = open(os.path.join(ref, "example/paddle-mnist.yaml"), "rb").read()
    return {"json_fields": sorted(tags), "string_constants": sorted(consts), "flags": sorted(flags),
            "example_paddle_mnist_sha256": hashlib.sha256(example).hexdigest()}


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    with open(OUT, "w") as fh:
        json.dump(record(sys.argv[1]), fh, indent=1, sort_keys=True)
        fh.write("\n")
    print("wrote", OUT)
