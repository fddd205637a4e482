"""What the reference (BitMapperBS) writes for the inputs of the tests that compare with it, kept as sha256 digests in
tests/golden/reference_sha256.json, so that those comparisons run where the reference is not built (oracle/build_ref.sh
needs its sources).  Where it is built, the tests compare with it directly as well.

The digests were recorded from this project's output at a commit whose tests had found that output identical to the
reference's, byte for byte, on the same seeded inputs.  To record them again (after a deliberate change of the inputs),
run the tests with BMBS_RECORD_SHA256=<file>: check() then appends one {key: digest} line per call to <file> instead of
comparing."""
import hashlib
import json
import os
from pathlib import Path

FILE = Path(__file__).resolve().parent / "golden" / "reference_sha256.json"


def check(key: str, data: bytes):
    got = hashlib.sha256(data).hexdigest()
    record = os.environ.get("BMBS_RECORD_SHA256")
    if record:
        with open(record, "a") as f:
            f.write(json.dumps({key: got}) + "\n")
        return
    want = json.loads(FILE.read_text()).get(key)
    assert want is not None, f"no stored digest for {key} in {FILE.name}"
    assert got == want, f"{key}: output differs from the reference's (sha256 {got}, stored {want})"
