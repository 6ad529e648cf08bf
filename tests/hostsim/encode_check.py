"""TEST INFRASTRUCTURE ONLY: round-trip check of the device encoder sources (csrc/ck_lz4_enc.cuh, csrc/ck_deflate.cuh)
built with g++ under AddressSanitizer / UBSan (tests/hostsim/encoders.cpp).  Every gzip member must decode to its input
under zlib and under the host build of the device decoder (ck_gunzip); every LZ4 frame under the LZ4 restatement
(tests/golden/kafka_codecs.py), the host build of the device decoder (ck_lz4_frame) and the system liblz4 where it loads.

    python tests/hostsim/encode_check.py --lib PATH [--random N] [--seed S]

must run with the sanitizer runtime preloaded (see run()); prints one JSON line of totals and exits non-zero on the first
disagreement.  A sanitizer report aborts the process."""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import random
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(ROOT, "calfkit-sdk_b200", "csrc")
for p in (ROOT, os.path.join(ROOT, "calfkit-sdk_b200"), os.path.join(ROOT, "tests", "golden"), HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

import kafka_codecs as kc  # noqa: E402
from codec_check import Codecs  # noqa: E402

GZIP, LZ4 = 1, 3


def build(out_dir: str) -> str:
    lib = os.path.join(out_dir, "libck_encoders_hostsim.so")
    subprocess.check_call(["g++", "-O1", "-g", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas",
                           "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined", "-I", CSRC, "-o", lib,
                           os.path.join(HERE, "encoders.cpp")])
    return lib


def run(args: list[str], timeout: float = 900) -> subprocess.CompletedProcess:
    """build into a temporary directory and run this module with the sanitizer runtimes preloaded"""
    with tempfile.TemporaryDirectory() as d:
        lib = build(d)
        pre = [subprocess.check_output(["g++", f"-print-file-name={n}"], text=True).strip() for n in ("libasan.so", "libubsan.so")]
        env = dict(os.environ, LD_PRELOAD=" ".join(pre), ASAN_OPTIONS="detect_leaks=0:abort_on_error=0:exitcode=99",
                   UBSAN_OPTIONS="print_stacktrace=1:halt_on_error=1:exitcode=98", PYTHONDONTWRITEBYTECODE="1")
        return subprocess.run([sys.executable, os.path.abspath(__file__), "--lib", lib] + args, env=env, capture_output=True,
                              text=True, timeout=timeout)


class Encoders(Codecs):
    def __init__(self, path: str):
        super().__init__(path)
        self.L.ck_host_encode.argtypes = [ctypes.c_char_p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_uint64]
        self.L.ck_host_encode.restype = ctypes.c_uint64
        self.L.ck_host_enc_bound.argtypes = [ctypes.c_uint32, ctypes.c_uint32]
        self.L.ck_host_enc_bound.restype = ctypes.c_uint64

    def encode(self, data: bytes, codec: int) -> bytes:
        cap = self.L.ck_host_enc_bound(len(data), codec)
        out = ctypes.create_string_buffer(max(cap, 1))
        n = self.L.ck_host_encode(data, len(data), codec, out, cap)
        assert n, "encoder refused a buffer of the stated worst-case size"
        return out.raw[:n]


def lz4_blocks(frame: bytes) -> list[tuple[bool, int]]:
    """(raw, size) of every block of a frame written with FLG 0x60"""
    pos, out = 7, []
    while True:
        bs = int.from_bytes(frame[pos:pos + 4], "little")
        pos += 4
        if not bs:
            return out
        out.append((bool(bs >> 31), bs & 0x7FFFFFFF))
        pos += bs & 0x7FFFFFFF


class Checker:
    def __init__(self, enc: Encoders):
        self.e, self.lib = enc, kc.liblz4()
        self.tot = {"inputs": 0, "bytes": 0, "gzip_bytes": 0, "lz4_bytes": 0, "liblz4": 0, "raw_lz4_inputs": 0,
                    "stored_deflate_inputs": 0}

    def check(self, data: bytes, what) -> tuple[bytes, bytes]:
        g, f = self.e.encode(data, GZIP), self.e.encode(data, LZ4)
        bound = self.e.L.ck_host_enc_bound(len(data), GZIP), self.e.L.ck_host_enc_bound(len(data), LZ4)
        assert len(g) <= bound[0] and len(f) <= bound[1], ("bound", what)
        assert g[:10] == bytes.fromhex("1f8b08000000000000ff") and g[-10:-8] == b"\x03\x00", ("gzip framing", what)
        assert f[:7] == bytes.fromhex("04224d18604082") and f[-4:] == b"\0\0\0\0", ("lz4 framing", what)
        assert kc.gzip_decode(g) == data, ("zlib", what)
        assert self.e.gunzip(g) == data, ("ck_gunzip", what)
        assert kc.lz4_frame_decode(f) == data, ("restated lz4", what)
        assert self.e.lz4(f) == data, ("ck_lz4_frame", what)
        if self.lib is not None:
            assert kc.liblz4_decompress(self.lib, f, len(data)) == data, ("liblz4", what)
            self.tot["liblz4"] += 1
        self.tot["inputs"] += 1
        self.tot["bytes"] += len(data)
        self.tot["gzip_bytes"] += len(g)
        self.tot["lz4_bytes"] += len(f)
        return g, f


def record_sections(rng: random.Random) -> list[bytes]:
    from calfkit import synth
    from oracle import kafka_batch as kb
    fx = kc.load_fixture(os.path.join(ROOT, "tests", "golden", "kafka_codecs.json"))
    out = [plain for _c, _f, plain in fx]
    recs = synth.tool_events(600, seed=rng.randrange(1 << 30)) + synth.tool_events(40, seed=5, size=None, full_history=True)
    krecs = [kb.calfkit_record(r, f"{i:032x}") for i, r in enumerate(recs)]
    for lo, hi in ((0, 14), (14, 70), (70, 640)):
        out.append(kc.records_section(krecs[lo:hi]))
    return out


def mixture(rng: random.Random) -> bytes:
    words = [b'{"ctx":', b'"correlation_id"', b"get_weather", b"It's sunny in ", b'"location":', b"Paris", b",", b"}", b"\n"]
    n = rng.choice([0, 1, 3, 7, 12, 13, 16, 31, 64, 100, 300, 700, 1500, 3000])
    out = bytearray()
    while len(out) < n:
        k = rng.randrange(5)
        if k == 0:
            out += bytes(rng.randrange(256) for _ in range(rng.randrange(1, 20)))
        elif k == 1:
            out += bytes([rng.randrange(256)]) * rng.randrange(1, 300)
        elif k == 2 and out:
            s = rng.randrange(len(out))
            out += out[s:s + rng.randrange(1, 300)]
        else:
            out += rng.choice(words)
    return bytes(out[:n])


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", required=True)
    ap.add_argument("--random", type=int, default=2000)
    ap.add_argument("--seed", type=int, default=1)
    a = ap.parse_args()
    ch = Checker(Encoders(a.lib))
    rng = random.Random(a.seed)
    fixed = [b""] + [bytes(rng.randrange(256) for _ in range(n)) for n in range(1, 65)] + [b"ab" * n for n in range(1, 33)]
    text = b"".join(rng.choice([b'{"location":"Paris"}', b"It's sunny in ", b"get_weather", b"0123456789abcdef"]) for _ in range(9000))
    for n in (65535, 65536, 65537):
        fixed += [text[:n], bytes(n)]
    for period in (1, 2, 3):
        unit = bytes(rng.randrange(256) for _ in range(period))
        fixed += [unit * (n // period) for n in (20, 4096, 70000, 200000)]
    for i, d in enumerate(fixed):
        ch.check(d, ("fixed", i, len(d)))
    for n in (1000, 65536, 65537, 300000):                      # incompressible: raw LZ4 blocks, stored DEFLATE blocks
        d = bytes(rng.randrange(256) for _ in range(n))
        g, f = ch.check(d, ("random bytes", n))
        assert all(raw for raw, _ in lz4_blocks(f)), ("random bytes must give raw LZ4 blocks", n)
        assert (g[10] >> 1) & 3 == 0, ("random bytes must give stored DEFLATE blocks", n)
        ch.tot["raw_lz4_inputs"] += 1
        ch.tot["stored_deflate_inputs"] += 1
    for i, d in enumerate(record_sections(rng)):
        ch.check(d, ("records section", i, len(d)))
    for i in range(a.random):
        ch.check(mixture(rng), ("mixture", i))
    print(json.dumps(ch.tot))
    return 0


if __name__ == "__main__":
    sys.exit(main())
