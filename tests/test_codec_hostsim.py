"""The device decoders of compressed Kafka record batches (csrc/ck_inflate.cuh, csrc/ck_lz4.cuh) compiled with g++ under
AddressSanitizer and UBSan in their own library (tests/hostsim/codecs.cpp), checked on the CPU against zlib and the LZ4
restatement: every fixture frame byte-exact, 100 K random zlib streams (random levels, strategies and memLevels)
byte-exact, restated LZ4 frames over the option matrix, and mutated gzip / LZ4 streams either rejected or accepted with
exactly the bytes zlib (or the LZ4 restatement) produces.  scripts/fuzz_codecs.py runs larger counts."""
import json
import os
import shutil
import sys

import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostsim"))


@pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++")
def test_codecs_under_sanitizers():
    import codec_check
    r = codec_check.run(["--small", "100000", "--random", "800", "--mutations", "2000", "--seed", "20261017"])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-6000:]
    assert "ERROR: AddressSanitizer" not in r.stderr and "runtime error" not in r.stderr, r.stderr[-6000:]
    tot = json.loads(r.stdout.strip().splitlines()[-1])
    assert tot["fixtures"] >= 35 and tot["zlib_streams"] >= 100000 and tot["lz4_frames"] >= 100
    assert tot["gzip_mutants"] == 2000 and tot["lz4_mutants"] == 2000
