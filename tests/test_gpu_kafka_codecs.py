"""Compressed Kafka record batches on the device: frames whose records section is gzip (codec 1) or LZ4 (codec 3) are
decompressed by csrc/ck_inflate.cuh / csrc/ck_lz4.cuh into slots after the submitted bytes, and the split, field decode,
walk, plan and emit read them there.  Expectations come from the CPU restatement (tests/golden/kafka_codecs.py: zlib and the
restated LZ4 frame format) and from fixture frames written by zlib and liblz4 (tests/golden/kafka_codecs.json)."""
import json
import os
import struct

import numpy as np
import pytest

import kafka_codecs as kc
from oracle import kafka_batch as kb

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture()
def engine():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from calfkit.engine import BatchEngine, ToolTemplate
    e = BatchEngine(0, max_records=1 << 17, max_in_bytes=256 << 20)
    e.register_topics(["tool.get_weather.input", "tool.get_weather.output", "weather_agent.input"], num_partitions=8)
    e.set_tool_node("tool.get_weather.output", ToolTemplate.from_format("It's sunny in {location}"))
    yield e
    e.close()


def u8(b: bytes) -> np.ndarray:
    return np.frombuffer(b, dtype=np.uint8)


def check_index(engine, krecs, bad=None):
    """every record's value / key / correlation_id header, read through rb_index() and the host view, equals krecs"""
    ix, data = engine.rb_index(), engine.rb_bytes()
    want_bad = np.zeros(len(krecs), np.uint32) if bad is None else bad
    assert len(ix["bad"]) == len(krecs)
    assert (ix["bad"] == want_bad).all(), np.nonzero(ix["bad"] != want_bad)[0][:10]
    for i, k in enumerate(krecs):
        if want_bad[i]:
            continue
        assert data[ix["val_off"][i]:ix["val_off"][i] + ix["val_len"][i]].tobytes() == k.value, i
        assert (ix["key_len"][i] == -1) == (k.key is None), i
        if k.key is not None:
            assert data[ix["key_off"][i]:ix["key_off"][i] + ix["key_len"][i]].tobytes() == k.key, i
        assert data[ix["corr_off"][i]:ix["corr_off"][i] + ix["corr_len"][i]].tobytes() == dict(k.headers)["correlation_id"], i


def fixture_frames():
    return [(c["name"], frame, kb.decode_batches(kc.frame_with_section(plain, kc.NONE, c["records"])))
            for c, frame, plain in kc.load_fixture(os.path.join(HERE, "golden", "kafka_codecs.json"))]


def test_fixture_frames_alone_and_together(engine):
    frames = fixture_frames()
    for name, frame, krecs in frames:
        assert engine.submit_recordbatch(u8(frame)) == len(krecs), name
        check_index(engine, krecs)
    buf = b"".join(f for _n, f, _k in frames)
    allrecs = [k for _n, _f, ks in frames for k in ks]
    assert engine.submit_recordbatch(u8(buf)) == len(allrecs)
    check_index(engine, allrecs)
    assert len(engine.rb_decompressed()) >= sum(len(kc.records_section(ks)) for _n, _f, ks in frames)


# codecs of the mixed fetch, cycled over its frames
MIXED = [None, ("gzip", dict(level=0)), ("gzip", dict(level=1)), ("gzip", dict(level=6, fname=b"r.bin")), ("gzip", dict(level=9)),
         ("lz4", dict(linked=False)), ("lz4", dict(linked=True, content_size=True)), ("lz4", dict(block_checksum=True, content_checksum=False)),
         ("lz4", dict(linked=True, block_checksum=True, content_checksum=True, raw_blocks="odd")), ("lz4", dict(block_size_id=7)),
         ("lz4", dict(block_size_id=4, raw_blocks="all"))]


def mixed_fetch(recs, sizes, codecs):
    out, krecs, k = [], [], 0
    for bi, sz in enumerate(sizes):
        chunk = [kb.calfkit_record(r, json.loads(r)["context"]["deps"]["correlation_id"], keyed=j % 4 != 0) for j, r in enumerate(recs[k:k + sz])]
        c = codecs[bi % len(codecs)]
        f = kc.encode_batch(chunk, base_offset=1000 + k, base_timestamp=1767225600000 + bi, compression=c and c[0], **(c[1] if c else {}))
        out.append(f)
        krecs += chunk
        k += sz
    return out, krecs


def test_mixed_fetch_feeds_the_walker(engine):
    import tools_def
    from calfkit import synth
    from calfkit.engine._lib import CK_OK, COL
    from oracle import port
    recs = (synth.tool_events(1500, seed=81) + synth.tool_events(200, seed=82, size=None, full_history=True)
            + synth.mixed_events(60, seed=83, lo=20000, hi=30000))                         # 30 KB records cross 64 KB LZ4 blocks
    sizes = [1, 14, 14, 200, 3, 500, 700, 268, 20, 20, 1, 19]
    assert sum(sizes) == len(recs)
    frames, krecs = mixed_fetch(recs, sizes, MIXED)
    buf = b"".join(frames) + frames[3][:45]                                               # a truncated tail
    assert [r.value for r in kc.decode_batches(buf)] == recs
    assert engine.submit_recordbatch(u8(buf)) == len(recs)
    check_index(engine, krecs)
    engine.tool_plan()
    out = engine.fetch()
    assert (out.cols[COL["STATUS"]] == CK_OK).all()
    node = port.ToolNode.of(tools_def.get_weather)
    got = [(p.topic, p.key, p.payload) for p in out.publishes()]
    assert got == [(t, k, pl) for r in recs for (t, k, _c, pl) in port.tool_node_event(node, r)]


def _reframe(frame: bytes, section: bytes, count: int | None = None) -> bytes:
    """the same frame with another records section (and recordsCount), CRC32C recomputed: only the codec can notice"""
    codec = struct.unpack_from(">h", frame, kb.CRC_FROM)[0] & 7
    n = struct.unpack_from(">i", frame, 57)[0] if count is None else count
    return kc.frame_with_section(section, codec, n, base_offset=struct.unpack_from(">q", frame, 0)[0])


def _lz4_frame(block: bytes, flg: int = 0x60) -> bytes:
    desc = bytes([flg, 0x40])
    return struct.pack("<I", kc.LZ4_MAGIC) + desc + bytes([(kc.xxh32(desc) >> 8) & 0xFF]) + struct.pack("<I", len(block)) + block + b"\0\0\0\0"


def damaged(recs):
    """(name, frame) pairs: compressed records sections damaged in one way each"""
    g = kc.encode_batch(recs, compression="gzip", level=6)
    gs = g[kb.HEADER_LEN:]
    plain = kc.records_section(recs)
    out = []
    m = bytearray(gs); m[len(m) // 2] ^= 0x10; out.append(("gzip bit flip", _reframe(g, bytes(m))))
    m = bytearray(gs); m[-8] ^= 1; out.append(("gzip CRC-32", _reframe(g, bytes(m))))
    m = bytearray(gs); m[-4] ^= 1; out.append(("gzip ISIZE", _reframe(g, bytes(m))))
    out.append(("gzip truncated", _reframe(g, gs[:len(gs) - 20] + gs[-8:])))
    out.append(("gzip trailing bytes", _reframe(g, gs + b"\x1f\x8b")))
    out.append(("gzip second member", _reframe(g, gs + kc.gzip_encode(b""))))
    lz = kc.encode_batch(recs, compression="lz4", block_checksum=True, content_checksum=True)
    ls = lz[kb.HEADER_LEN:]
    out.append(("lz4 offset 0", _reframe(lz, _lz4_frame(bytes([0x40]) + plain[:4] + b"\0\0" + bytes([0x10]) + plain[4:5]))))
    out.append(("lz4 offset before start", _reframe(lz, _lz4_frame(bytes([0x40]) + plain[:4] + b"\x05\0" + bytes([0x10]) + plain[4:5]))))
    out.append(("lz4 literal past block", _reframe(lz, _lz4_frame(bytes([0xF0, 40]) + plain[:20]))))
    bs = struct.unpack_from("<I", ls, 7)[0] & 0x7FFFFFFF
    m = bytearray(ls); m[11 + bs] ^= 1; out.append(("lz4 block checksum", _reframe(lz, bytes(m))))
    m = bytearray(ls); m[-1] ^= 1; out.append(("lz4 content checksum", _reframe(lz, bytes(m))))
    m = bytearray(ls); m[6] ^= 1; out.append(("lz4 header checksum", _reframe(lz, bytes(m))))
    desc = bytes([ls[4] | 1, ls[5]]) + b"\1\2\3\4"
    out.append(("lz4 DictID", _reframe(lz, ls[:4] + desc + bytes([(kc.xxh32(desc) >> 8) & 0xFF]) + ls[7:])))
    out.append(("recordsCount", _reframe(g, gs, count=len(recs) + 1)))
    out.append(("recordsCount lz4", _reframe(lz, ls, count=len(recs) - 1)))
    return out


def test_damaged_payloads_only_their_frame_is_bad(engine):
    from calfkit import synth
    from calfkit.engine._lib import CK_BAD_FRAME, CK_OK, COL
    import tools_def
    from oracle import port
    recs = synth.tool_events(40 * 17, seed=91)
    node = port.ToolNode.of(tools_def.get_weather)
    bad_recs = [kb.calfkit_record(r, json.loads(r)["context"]["deps"]["correlation_id"]) for r in recs[:20]]
    for name, bad in damaged(bad_recs):
        good, krecs = mixed_fetch(recs[20:100], [30, 50], [("gzip", {}), ("lz4", dict(linked=True))])
        buf = good[0] + bad + good[1]
        n = engine.submit_recordbatch(u8(buf))
        nbad = struct.unpack_from(">i", bad, 57)[0]
        assert n == 80 + nbad, name
        want = np.zeros(n, np.uint32); want[30:30 + nbad] = 1
        check_index(engine, krecs[:30] + [None] * nbad + krecs[30:], want)
        engine.tool_plan()
        out = engine.fetch()
        st = out.cols[COL["STATUS"]]
        assert (st[30:30 + nbad] == CK_BAD_FRAME).all() and (np.delete(st, np.s_[30:30 + nbad]) == CK_OK).all(), name
        got = [(p.topic, p.key, p.payload) for p in out.publishes()]
        assert got == [(t, k, pl) for r in recs[20:100] for (t, k, _c, pl) in port.tool_node_event(node, r)], name


def test_codecs_not_decoded_on_the_device(engine):
    from calfkit import synth
    recs = synth.tool_events(30, seed=93)
    frames, krecs = mixed_fetch(recs, [10, 10, 10], [("gzip", {})])
    sec = kc.records_section(krecs[10:20])
    for codec in (kc.SNAPPY, kc.ZSTD, 5, 6, 7):
        buf = frames[0] + kc.frame_with_section(sec, codec, 10) + frames[2]
        assert engine.submit_recordbatch(u8(buf)) == 30
        want = np.zeros(30, np.uint32); want[10:20] = 2
        check_index(engine, krecs, want)


def test_decompressed_size_over_max_in_bytes(engine):
    from calfkit import synth
    from calfkit.engine import BatchEngine
    from calfkit.exceptions import EngineError
    small = BatchEngine(0, max_records=4096, max_in_bytes=1 << 20)
    try:
        recs = synth.tool_events(1500, seed=95)
        frames, _ = mixed_fetch(recs, [1500], [("gzip", dict(level=9))])
        assert len(frames[0]) < (1 << 20) < len(kc.records_section([kb.KRecord(r) for r in recs]))
        with pytest.raises(EngineError, match="max_in_bytes"):
            small.submit_recordbatch(u8(frames[0]))
        frames, krecs = mixed_fetch(recs[:100], [60, 40], [("lz4", {}), ("gzip", {})])
        assert small.submit_recordbatch(u8(b"".join(frames))) == 100
        check_index(small, krecs)
    finally:
        small.close()


@pytest.mark.parametrize("codec", ["gzip", "lz4"])
@pytest.mark.parametrize("frame_bytes", [16 << 10, 1 << 20])
def test_64ki_records(engine, codec, frame_bytes):
    """65536 records (about 70 MB decompressed): frames built once for 4096 records and tiled, baseOffset rewritten"""
    from calfkit import synth
    recs = synth.tool_events(4096, seed=97)
    krecs = [kb.calfkit_record(r, json.loads(r)["context"]["deps"]["correlation_id"], keyed=i % 4 != 0) for i, r in enumerate(recs)]
    frames, chunk, size = [], [], 0
    for k in krecs + [None]:
        if k is None or (chunk and size + len(k.value) > frame_bytes):
            opts = dict(level=1) if codec == "gzip" else dict(linked=frame_bytes > 65536, content_size=True)
            frames.append(kc.encode_batch(chunk, compression=codec, **opts))
            chunk, size = [], 0
        if k is not None:
            chunk.append(k); size += len(k.value) + 100
    for f in frames:
        g = kb.decode_batches(kc.frame_with_section(kc.decompress_section(kc.GZIP if codec == "gzip" else kc.LZ4, f[kb.HEADER_LEN:]), 0,
                                                    struct.unpack_from(">i", f, 57)[0]))
        assert len(g) == struct.unpack_from(">i", f, 57)[0]
    tiled = bytearray()
    for t in range(16):
        for f in frames:
            g = bytearray(f); struct.pack_into(">q", g, 0, t * 4096); tiled += g
    assert engine.submit_recordbatch(u8(bytes(tiled))) == 65536
    check_index(engine, krecs * 16)
