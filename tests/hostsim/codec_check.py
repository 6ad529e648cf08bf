"""TEST INFRASTRUCTURE ONLY: differential check of the device codec sources (csrc/ck_inflate.cuh, csrc/ck_lz4.cuh) built
with g++ under AddressSanitizer / UBSan (tests/hostsim/codecs.cpp), against zlib and the LZ4 restatement
(tests/golden/kafka_codecs.py).

    python tests/hostsim/codec_check.py --lib PATH [--random N] [--mutations M] [--seed S]

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
import zlib

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(ROOT, "calfkit-sdk_b200", "csrc")
for p in (ROOT, os.path.join(ROOT, "tests", "golden")):
    if p not in sys.path:
        sys.path.insert(0, p)

import kafka_codecs as kc  # noqa: E402

STRATEGIES = [zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED]


def build(out_dir: str) -> str:
    lib = os.path.join(out_dir, "libck_codecs_hostsim.so")
    subprocess.check_call(["g++", "-O1", "-g", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas",
                           "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined", "-I", CSRC, "-o", lib,
                           os.path.join(HERE, "codecs.cpp")])
    return lib


def run(args: list[str], timeout: float = 600) -> subprocess.CompletedProcess:
    """build into a temporary directory and run this module with the sanitizer runtimes preloaded"""
    with tempfile.TemporaryDirectory() as d:
        lib = build(d)
        pre = [subprocess.check_output(["g++", f"-print-file-name={n}"], text=True).strip() for n in ("libasan.so", "libubsan.so")]
        env = dict(os.environ, LD_PRELOAD=" ".join(pre), ASAN_OPTIONS="detect_leaks=0:abort_on_error=0:exitcode=99",
                   UBSAN_OPTIONS="print_stacktrace=1:halt_on_error=1:exitcode=98", PYTHONDONTWRITEBYTECODE="1")
        return subprocess.run([sys.executable, os.path.abspath(__file__), "--lib", lib] + args, env=env, capture_output=True,
                              text=True, timeout=timeout)


class Codecs:
    def __init__(self, path: str):
        L = self.L = ctypes.CDLL(path)
        b, u32 = ctypes.c_char_p, ctypes.c_uint32
        for name, args in (("ck_host_gunzip", [b, u32, ctypes.c_void_p, u32]), ("ck_host_gzip_isize", [b, u32, ctypes.POINTER(u32)]),
                           ("ck_host_lz4_size", [b, u32, ctypes.POINTER(u32)]), ("ck_host_lz4_decode", [b, u32, ctypes.c_void_p, u32])):
            getattr(L, name).argtypes = args
            getattr(L, name).restype = ctypes.c_int

    def gunzip(self, src: bytes) -> bytes | None:
        """what the device does with a gzip records section: size from ISIZE, then inflate into exactly that slot"""
        isize = ctypes.c_uint32(0)
        if not self.L.ck_host_gzip_isize(src, len(src), ctypes.byref(isize)):
            return None
        out = ctypes.create_string_buffer(max(isize.value, 1))
        return out.raw[:isize.value] if self.L.ck_host_gunzip(src, len(src), out, isize.value) else None

    def lz4(self, src: bytes) -> bytes | None:
        """size pass, then decode into exactly that slot"""
        size = ctypes.c_uint32(0)
        if not self.L.ck_host_lz4_size(src, len(src), ctypes.byref(size)):
            return None
        out = ctypes.create_string_buffer(max(size.value, 1))
        return out.raw[:size.value] if self.L.ck_host_lz4_decode(src, len(src), out, size.value) else None


def _zlib_gunzip(src: bytes) -> bytes | None:
    try:
        return kc.gzip_decode(src)
    except Exception:
        return None


def _ref_lz4(src: bytes) -> bytes | None:
    try:
        return kc.lz4_frame_decode(src)
    except Exception:
        return None


def plaintext(rng: random.Random) -> bytes:
    """records-like text, runs, random bytes, and empty inputs"""
    kind = rng.randrange(6)
    n = rng.choice([0, 1, 5, 17, 100, 1000, 5000, 40000]) if kind else 0
    if kind == 1:
        return bytes(rng.randrange(256) for _ in range(n))
    if kind == 2:
        return bytes([rng.randrange(4)]) * n
    words = [b'{"ctx":', b'"correlation_id"', b"get_weather", b"It's sunny in ", b'"location":', b"Paris", b",", b"}", b"\n"]
    out = bytearray()
    while len(out) < n:
        out += rng.choice(words) if rng.random() < 0.9 else bytes([rng.randrange(256)])
    return bytes(out[:n])


def mutate(rng: random.Random, b: bytes) -> bytes:
    m = bytearray(b)
    k = rng.randrange(4)
    if k == 0 or not m:
        m += bytes(rng.randrange(256) for _ in range(rng.randrange(1, 4)))
    elif k == 1:
        del m[rng.randrange(len(m)):]
    else:
        for _ in range(rng.randrange(1, 4)):
            i = rng.randrange(len(m))
            m[i] ^= 1 << rng.randrange(8) if k == 2 else rng.randrange(1, 256)
    return bytes(m)


def check_fixtures(c: Codecs, path: str) -> int:
    cases = kc.load_fixture(path)
    for case, frame, plain in cases:
        got = c.gunzip(frame[61:]) if case["codec"] == "gzip" else c.lz4(frame[61:])
        assert got == plain, f"fixture {case['name']}"
    return len(cases)


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", required=True)
    ap.add_argument("--random", type=int, default=1000)
    ap.add_argument("--mutations", type=int, default=1000)
    ap.add_argument("--small", type=int, default=0, help="short random zlib streams (random level, strategy, memLevel)")
    ap.add_argument("--seed", type=int, default=1)
    a = ap.parse_args()
    c = Codecs(a.lib)
    rng = random.Random(a.seed)
    tot = {"fixtures": check_fixtures(c, os.path.join(ROOT, "tests", "golden", "kafka_codecs.json")), "zlib_streams": 0,
           "lz4_frames": 0, "gzip_mutants": 0, "gzip_mutants_accepted": 0, "lz4_mutants": 0, "lz4_mutants_accepted": 0}
    texts = [plaintext(rng) for _ in range(64)]
    for i in range(a.random):
        p = rng.choice(texts) if i % 4 else plaintext(rng)
        g = kc.gzip_encode(p, level=rng.randrange(10), strategy=rng.choice(STRATEGIES), mem_level=rng.randrange(1, 10))
        assert c.gunzip(g) == p, ("zlib stream", i)
        tot["zlib_streams"] += 1
        if i % 8 == 0:
            f = kc.lz4_frame_encode(p[:20000], block_size_id=rng.randrange(4, 8), linked=rng.random() < 0.5,
                                    block_checksum=rng.random() < 0.5, content_size=rng.random() < 0.5,
                                    content_checksum=rng.random() < 0.5, raw_blocks=rng.choice(["auto", "odd"]))
            assert c.lz4(f) == p[:20000], ("lz4 frame", i)
            tot["lz4_frames"] += 1
    for i in range(a.small):
        n = rng.choice([0, 1, 3, 30, 200, 700, 1500])
        p = bytes(rng.randrange(4) + 97 for _ in range(n)) if i % 3 else rng.choice(texts)[:n]
        g = kc.gzip_encode(p, level=rng.randrange(10), strategy=rng.choice(STRATEGIES), mem_level=rng.randrange(1, 10))
        assert c.gunzip(g) == p, ("short zlib stream", i, g.hex())
        tot["zlib_streams"] += 1
    for i in range(a.mutations):
        p = rng.choice(texts)
        g = mutate(rng, kc.gzip_encode(p, level=rng.randrange(10), strategy=rng.choice(STRATEGIES)))
        got = c.gunzip(g)
        tot["gzip_mutants"] += 1
        if got is not None:                     # accepted: CRC-32 and ISIZE passed, so it must be what zlib makes of it
            tot["gzip_mutants_accepted"] += 1
            want = _zlib_gunzip(g)
            assert got == (want if want is not None else p), ("gzip mutant", i, g.hex())
        f = mutate(rng, kc.lz4_frame_encode(p, block_size_id=4, linked=i % 2 == 0, block_checksum=i % 3 == 0,
                                            content_size=i % 5 == 0, content_checksum=i % 7 != 0))
        got, want = c.lz4(f), _ref_lz4(f)
        tot["lz4_mutants"] += 1
        tot["lz4_mutants_accepted"] += got is not None
        assert got == want, ("lz4 mutant", i, f.hex())
    print(json.dumps(tot))
    return 0


if __name__ == "__main__":
    sys.exit(main())
