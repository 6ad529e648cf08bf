"""Larger runs of the codec differential check (tests/test_codec_hostsim.py runs a bounded one): the device gzip and LZ4
decoders built with g++ under AddressSanitizer / UBSan against zlib and the LZ4 restatement.

    python scripts/fuzz_codecs.py [--small 2000000] [--random 20000] [--mutations 200000] [--seed 1]
"""
import argparse
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "hostsim"))
sys.dont_write_bytecode = True

import codec_check  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--small", type=int, default=2000000)
ap.add_argument("--random", type=int, default=20000)
ap.add_argument("--mutations", type=int, default=200000)
ap.add_argument("--seed", type=int, default=1)
a = ap.parse_args()
r = codec_check.run(["--small", str(a.small), "--random", str(a.random), "--mutations", str(a.mutations), "--seed", str(a.seed)],
                    timeout=24 * 3600)
print(r.stdout, end="")
if r.returncode:
    print(r.stderr[-8000:], file=sys.stderr)
sys.exit(r.returncode)
