"""API-surface parity with the reference, checked mechanically against a recording of its sources
(``tests/golden/reference_api.json``, written by ``tools/record_reference_api.py``): every JSON field of its Go API types,
every string constant of its API package and every command-line flag of its options exists here under the same spelling."""
import dataclasses
import hashlib
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_api.json")))


def test_every_json_field_of_the_reference_api_types_exists():
    """types.go:29-152, replica.go:9-63 -- byte-compatible spellings incl. ``RestartCount`` and phase ``Succeed``."""
    from trainingjob_operator_b200.api import types as T

    tags = set(REF["json_fields"])
    ours = set()
    for name in dir(T):
        c = getattr(T, name)
        if dataclasses.is_dataclass(c):
            ours |= {f.metadata.get("json", f.name) for f in dataclasses.fields(c)}
    assert len(tags) >= 40 and not (tags - ours), sorted(tags - ours)


def test_every_string_constant_of_the_reference_api_package_exists():
    ref = set(REF["string_constants"])
    ours = open(os.path.join(ROOT, "trainingjob_operator_b200/api/constants.py")).read() + \
        open(os.path.join(ROOT, "trainingjob_operator_b200/api/types.py")).read()
    missing = [c for c in sorted(ref) if f'"{c}"' not in ours and f"'{c}'" not in ours]
    assert len(ref) >= 45 and not missing, missing


def test_every_command_line_flag_of_the_reference_exists():
    """cmd/app/options/options.go:61-72 (+ the leader-election set bound by leaderelectionconfig.BindFlags)."""
    flags = set(REF["flags"])
    ours = open(os.path.join(ROOT, "trainingjob_operator_b200/cmd/options.py")).read()
    missing = [f for f in sorted(flags) if f"--{f}" not in ours and f'"{f}"' not in ours]
    assert len(flags) >= 9 and not missing, missing
    for f in ("leader-elect", "leader-elect-lease-duration", "leader-elect-renew-deadline", "leader-elect-retry-period"):
        assert f in ours, f


def test_the_reference_example_is_shipped_verbatim():
    ours = open(os.path.join(ROOT, "examples/paddle-mnist.yaml"), "rb").read()
    assert hashlib.sha256(ours).hexdigest() == REF["example_paddle_mnist_sha256"]
