"""Writes tests/golden/kafka_codecs.json: Kafka RecordBatch v2 frames whose records sections were compressed by real
compressors — zlib (every level 0-9 and the strategies FIXED / HUFFMAN_ONLY / RLE / FILTERED, in a gzip member whose header
carries FNAME and FEXTRA) and the system liblz4 (LZ4F_compressFrame over the frame option matrix: block maximum, linked /
independent blocks, block and content checksums, content size; incompressible records give uncompressed blocks).  Each
case stores the frame (its records section compressed) and names its plaintext records section in "plains" (stored
zlib-compressed to keep the file small).  Runs only where liblz4 loads:

    python tests/golden/make_golden_kafka_codecs.py
"""
import base64
import itertools
import json
import os
import random
import sys
import zlib

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (os.path.join(ROOT, "calfkit-sdk_b200"), ROOT, HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

import kafka_codecs as kc  # noqa: E402
from oracle import kafka_batch as kb  # noqa: E402


def records(n: int, distinct: int, seed: int, noise: int = 0) -> list:
    """n calfkit records cycling through `distinct` short ones, so that the frames stay small while the records sections
    of the LZ4 cases still span two 64 KB blocks; noise > 0: values of that many random bytes (raw LZ4 blocks)"""
    rng = random.Random(seed)
    base = []
    for i in range(distinct):
        corr = "%032x" % rng.getrandbits(128)
        value = bytes(rng.randrange(256) for _ in range(noise)) if noise else json.dumps(
            {"id": i, "tool": "get_weather", "args": {"location": rng.choice(["Paris", "Cairo", "Lima"])}, "corr": corr}).encode()
        base.append(kb.calfkit_record(value, corr, keyed=i % 4 != 0))
    return [base[i % distinct] for i in range(n)]


def main() -> None:
    lib = kc.liblz4()
    if lib is None:
        sys.exit("liblz4 not found: the fixture needs the system library")
    b64 = lambda b: base64.b64encode(b).decode()  # noqa: E731
    cases, plains = [], {}

    def add(name, codec, recs, section, base_offset):
        plain = b64(zlib.compress(kc.records_section(recs), 9))
        pid = plains.setdefault(plain, str(len(plains)))
        frame = kc.frame_with_section(section, codec, len(recs), base_offset=base_offset)
        cases.append({"name": name, "codec": {kc.GZIP: "gzip", kc.LZ4: "lz4"}[codec], "records": len(recs), "plain": pid,
                      "frame": b64(frame)})

    small = records(12, 12, seed=901)
    for level in range(10):
        add(f"gzip-level{level}", kc.GZIP, small, kc.gzip_encode(kc.records_section(small), level=level, fname=b"records.bin",
                                                                   fextra=b"ck\x04\x00test"), 100 + level)
    for sname in ("Z_FIXED", "Z_HUFFMAN_ONLY", "Z_RLE", "Z_FILTERED"):
        add(f"gzip-{sname}", kc.GZIP, small, kc.gzip_encode(kc.records_section(small), level=6, strategy=getattr(zlib, sname),
                                                             fname=b"r", fextra=b""), 200)
    big = records(320, 3, seed=902)                                   # > 64 KB of records: two blocks
    for linked, bsum, csize, csum in itertools.product((False, True), repeat=4):
        name = f"lz4-64KB-{'linked' if linked else 'indep'}{'-bsum' if bsum else ''}{'-csize' if csize else ''}{'-csum' if csum else ''}"
        add(name, kc.LZ4, big, kc.liblz4_compress(lib, kc.records_section(big), 4, linked, bsum, csize, csum), 300)
    for bid in (5, 6, 7):
        add(f"lz4-bsize{bid}-csum", kc.LZ4, big, kc.liblz4_compress(lib, kc.records_section(big), bid, False, False, True, True), 400 + bid)
    noisy = records(2, 2, seed=903, noise=1024)
    add("lz4-incompressible-blocks", kc.LZ4, noisy, kc.liblz4_compress(lib, kc.records_section(noisy), 4, False, True, False, True), 500)
    add("lz4-hc-linked", kc.LZ4, big, kc.liblz4_compress(lib, kc.records_section(big), 4, True, False, True, True, level=9), 600)
    head = {"generator": "tests/golden/make_golden_kafka_codecs.py", "zlib": zlib.ZLIB_RUNTIME_VERSION,
            "liblz4": lib.LZ4_versionNumber(), "plains": {v: k for k, v in plains.items()}}
    with open(os.path.join(HERE, "kafka_codecs.json"), "w") as f:      # one case per line
        f.write(json.dumps(head)[:-1] + ', "cases": [\n' + ",\n".join(json.dumps(c) for c in cases) + "]}\n")
    print(f"{len(cases)} cases")


if __name__ == "__main__":
    main()
