"""The device encoders of compressed Kafka record batches (csrc/ck_lz4_enc.cuh, csrc/ck_deflate.cuh) compiled with g++
under AddressSanitizer and UBSan in their own library (tests/hostsim/encoders.cpp) and run on the CPU: the empty input,
1-64 bytes, 64 KB +- 1, zeros, period-1/2/3 runs, random bytes (raw LZ4 blocks, stored DEFLATE blocks), the records
sections of the fixture and of synthetic tool events, and 20 K random mixtures.  Every gzip member must decode to its input
under zlib and under the host build of the device decoder; every LZ4 frame under the LZ4 restatement, the host build of
the device decoder and the system liblz4 where it loads; every section must stay within the worst-case size."""
import json
import os
import shutil
import sys

import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostsim"))


@pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++")
def test_encoders_under_sanitizers():
    import encode_check
    r = encode_check.run(["--random", "20000", "--seed", "20261017"])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-6000:]
    assert "ERROR: AddressSanitizer" not in r.stderr and "runtime error" not in r.stderr, r.stderr[-6000:]
    tot = json.loads(r.stdout.strip().splitlines()[-1])
    assert tot["inputs"] >= 20000 + 100 and tot["raw_lz4_inputs"] == 4 and tot["stored_deflate_inputs"] == 4
