"""The CPU restatement of the compressed Kafka record batches (tests/golden/kafka_codecs.py): it decodes the fixture frames
written by zlib and the system liblz4 (tests/golden/kafka_codecs.json) to their stored records, its own encoder's frames
decode back, and — where liblz4 loads — liblz4 accepts the restated encoder's frames."""
import itertools
import json
import os
import struct

import pytest

import kafka_codecs as kc
from oracle import kafka_batch as kb

HERE = os.path.dirname(os.path.abspath(__file__))


def fixture():
    return kc.load_fixture(os.path.join(HERE, "golden", "kafka_codecs.json"))


def plain_records(plain: bytes, count: int):
    return kb.decode_batches(kc.frame_with_section(plain, kc.NONE, count))


def test_fixture_covers_the_option_matrix():
    names = [c["name"] for c, _f, _p in fixture()]
    assert {f"gzip-level{k}" for k in range(10)} <= set(names)
    assert {"gzip-Z_FIXED", "gzip-Z_HUFFMAN_ONLY", "gzip-Z_RLE", "gzip-Z_FILTERED"} <= set(names)
    assert sum(n.startswith("lz4-64KB-") for n in names) == 16
    flags = {f[kb.HEADER_LEN + 4] for c, f, _p in fixture() if c["codec"] == "lz4"}
    assert len({x & 0x3C for x in flags}) == 16                 # independent, block checksum, content size, content checksum
    lz = {c["name"]: f[kb.HEADER_LEN:] for c, f, _p in fixture() if c["codec"] == "lz4"}
    assert lz["lz4-incompressible-blocks"][7 + 3] & 0x80        # an uncompressed block (bit 31 of its size)
    assert struct.unpack_from("<I", lz["lz4-64KB-linked"], 7)[0] < len(lz["lz4-64KB-linked"]) - 16   # more than one block


@pytest.mark.parametrize("i", range(35))
def test_oracle_decodes_fixture_frames(i):
    case, frame, plain = fixture()[i]
    assert kc.decompress_section({"gzip": kc.GZIP, "lz4": kc.LZ4}[case["codec"]], frame[kb.HEADER_LEN:]) == plain
    got = kc.decode_batches(frame)
    want = plain_records(plain, case["records"])
    assert len(got) == case["records"]
    assert [(r.value, r.key, r.headers) for r in got] == [(r.value, r.key, r.headers) for r in want]


def test_xxh32_known_answers():
    # the published XXH32 sanity values (seed 0): empty input and "a" / "abc"
    assert kc.xxh32(b"") == 0x02CC5D05
    assert kc.xxh32(b"a") == 0x550D7456
    assert kc.xxh32(b"abc") == 0x32D153FF
    # and liblz4's content checksums in the fixture are XXH32 of the plaintext
    n = 0
    for case, frame, plain in fixture():
        sec = frame[kb.HEADER_LEN:]
        if case["codec"] == "lz4" and sec[4] & 0x04:
            assert int.from_bytes(sec[-4:], "little") == kc.xxh32(plain)
            n += 1
    assert n >= 8


def _recs(n, seed):
    from calfkit import synth
    recs = synth.tool_events(n, seed=seed)
    return [kb.calfkit_record(r, json.loads(r)["context"]["deps"]["correlation_id"], keyed=i % 4 != 0) for i, r in enumerate(recs)]


LZ4_OPTIONS = [dict(block_size_id=b, linked=lk, block_checksum=bs, content_size=cs, content_checksum=cc, raw_blocks=rb)
               for (lk, bs, cs, cc), b, rb in zip(itertools.product((False, True), repeat=4), itertools.cycle((4, 5, 6, 7)),
                                                  itertools.cycle(("auto", "odd", "auto")))]


@pytest.mark.parametrize("opts", LZ4_OPTIONS)
def test_restated_lz4_encoder_roundtrip(opts):
    recs = _recs(70, seed=5)
    f = kc.encode_batch(recs, base_offset=7, compression="lz4", **opts)
    got = kc.decode_batches(f)
    assert [(r.value, r.key, r.headers, r.offset) for r in got] == [(r.value, r.key, r.headers, 7 + i) for i, r in enumerate(recs)]


@pytest.mark.parametrize("level,strategy", [(0, 0), (1, 0), (6, 0), (9, 0), (6, 1), (6, 2), (6, 3), (6, 4)])
def test_restated_gzip_encoder_roundtrip(level, strategy):
    recs = _recs(30, seed=6)
    f = kc.encode_batch(recs, compression="gzip", level=level, strategy=strategy, fname=b"x")
    assert [r.value for r in kc.decode_batches(f)] == [r.value for r in recs]


def test_snappy_and_zstd_raise():
    recs = _recs(3, seed=7)
    for codec in (kc.SNAPPY, kc.ZSTD, 7):
        f = kc.frame_with_section(kc.records_section(recs), codec, len(recs))
        with pytest.raises(ValueError):
            kc.decode_batches(f)


@pytest.mark.parametrize("opts", LZ4_OPTIONS)
def test_liblz4_accepts_restated_frames(opts):
    lib = kc.liblz4()
    if lib is None:
        pytest.skip("the system liblz4 is not available")
    plain = kc.records_section(_recs(70, seed=8))
    assert kc.liblz4_decompress(lib, kc.lz4_frame_encode(plain, **opts), len(plain)) == plain
