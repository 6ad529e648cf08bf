"""Runs of Kafka RecordBatch v2 frames built on the device (BatchEngine.encode_recordbatches): every (topic, partition)
group split to the producer's batch size, records sections compressed with gzip or LZ4.  Checked against the framing
restatement (oracle/kafka_batch.py), the codecs restated in tests/golden/kafka_codecs.py, zlib,
the producer split restated in tests/golden/kafka_split.py,
the system liblz4 where it loads, and the device's own consume path (submit_recordbatch)."""
import os
import random
import struct
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostsim"))

pytestmark = pytest.mark.gpu

TS = 1767225600123
CODECS = {None: 0, "gzip": 1, "lz4": 3}
OVERHEAD = {None: lambda p: 0, "gzip": lambda p: 20 + 10 * ((p + 65535) // 65536), "lz4": lambda p: 11 + 4 * ((p + 65535) // 65536)}


def _engine(max_records=1 << 15, max_in=64 << 20, partitions=8):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from calfkit.engine import BatchEngine
    e = BatchEngine(0, max_records=max_records, max_in_bytes=max_in)
    e.register_topics(["tool.get_weather.input", "tool.get_weather.output", "weather_agent.input"], num_partitions=partitions)
    return e


@pytest.fixture(scope="module")
def planned():
    """an engine holding a tool-node plan: keyed publishes to weather_agent.input (8 partitions), unkeyed ones to
    tool.get_weather.output; groups = the partitions in order, then the unkeyed publishes, then an empty group"""
    from calfkit import synth
    from calfkit.engine import ToolTemplate
    from calfkit.engine._lib import COL
    from oracle import kafka_batch as kb
    e = _engine()
    e.set_tool_node("tool.get_weather.output", ToolTemplate.from_format("It's sunny in {location}"))
    recs = synth.tool_events(3000, seed=81) + synth.tool_events(200, seed=82, size=None, full_history=True)
    b = synth.pack(recs)
    e.submit(b.data, b.offsets)
    e.tool_plan()
    out = e.fetch()
    live = out.pubs["payload"] != 0xFFFFFFFF
    tid, tid2 = e.topic_ids["weather_agent.input"], e.topic_ids["tool.get_weather.output"]
    groups = [np.nonzero(live & (out.pubs["topic_id"] == tid) & (out.pubs["partition"] == p))[0] for p in range(8)]
    groups += [np.nonzero(live & (out.pubs["topic_id"] == tid2))[0][:900], np.zeros(0, np.int64)]

    def krec(j):
        p = out.pubs[j]
        r = int(p["record"])
        corr = out.record_bytes(r)[int(out.cols[COL["CORR_OFF"], r]):][:int(out.cols[COL["CORR_LEN"], r])].tobytes().decode()
        return kb.calfkit_record(out.payload(int(p["payload"])), corr, keyed=bool(p["has_key"]))
    want = [[krec(int(j)) for j in g] for g in groups]
    yield e, groups, want
    e.close()


def _encode(e, groups, **kw):
    idx = np.concatenate(groups).astype(np.uint32)
    data, off, grp = e.encode_recordbatches(idx, group_sizes=[len(g) for g in groups], timestamp_ms=TS, **kw)
    return data.tobytes(), off, grp


def _frames(data, off):
    return [data[off[i]:off[i + 1]] for i in range(len(off) - 1)]


def _check_run(data, off, grp, want, limit, codec, base_offsets):
    """every frame against the oracle: the greedy split of each group, kb.encode_batch header fields, CRC32C, the section"""
    import kafka_codecs as kc
    import kafka_split as ks
    from oracle import kafka_batch as kb
    frames = _frames(data, off)
    expect = []
    for g, recs in enumerate(want):
        done = 0
        for chunk in ks.split_batches(recs, limit):
            expect.append((g, chunk, base_offsets[g] + done))
            done += len(chunk)
    assert len(frames) == len(expect) and list(grp) == [g for g, _c, _b in expect]
    lib = kc.liblz4()
    for f, (g, chunk, base) in zip(frames, expect):
        plain = kb.encode_batch(chunk, base_offset=base, base_timestamp=TS)
        if codec is None:
            assert f == plain
            continue
        assert struct.unpack_from(">I", f, 17)[0] == kb.crc32c(f[kb.CRC_FROM:])
        assert struct.unpack_from(">i", f, 8)[0] == len(f) - 12
        assert f[:8] + f[12:17] == plain[:8] + plain[12:17] and f[23:61] == plain[23:61]
        assert struct.unpack_from(">h", f, 21)[0] == CODECS[codec]
        sec = f[61:]
        assert kc.decompress_section(CODECS[codec], sec) == plain[61:]
        assert len(sec) <= len(plain) - 61 + OVERHEAD[codec](len(plain) - 61)
        if codec == "lz4":
            assert sec[4:7] == bytes([0x60, 0x40, 0x82])
            if lib is not None:
                assert kc.liblz4_decompress(lib, sec, len(plain)) == plain[61:]
        else:
            assert sec[:10] == bytes.fromhex("1f8b08000000000000ff")
    return frames, expect


@pytest.mark.parametrize("codec", [None, "gzip", "lz4"])
@pytest.mark.parametrize("limit", [62, 2000, 16384, 1 << 20])
def test_runs_match_the_oracle(planned, codec, limit):
    e, groups, want = planned
    base = [1000 * g + 7 for g in range(len(groups))]
    idx = np.concatenate(groups).astype(np.uint32)
    data, off, grp = e.encode_recordbatches(idx, group_sizes=[len(g) for g in groups], base_offsets=base, timestamp_ms=TS,
                                            compression_type=codec, max_batch_size=limit)
    _check_run(data.tobytes(), off, grp, want, limit, codec, base)


def test_one_frame_groups_equal_encode_recordbatch(planned):
    e, groups, _want = planned
    for g in (groups[0], groups[3], groups[8]):
        data, off, grp = e.encode_recordbatches(g, base_offsets=[5000], timestamp_ms=TS, max_batch_size=1 << 30)
        assert len(off) == 2 and list(grp) == [0]
        assert data.tobytes() == e.encode_recordbatch(g, base_offset=5000, timestamp_ms=TS).tobytes()


def test_round_trip_through_the_consume_path(planned):
    """the frames of every codec, concatenated, read back by submit_recordbatch: no bad record, and every record's value,
    key and correlation_id equal its publish's, in send order"""
    e, groups, want = planned
    runs = [_encode(e, groups, compression_type=c, max_batch_size=lim) for c in CODECS for lim in (16384, 1 << 20)]
    flat = [r for g in want for r in g]
    for data, _off, _grp in runs:
        n = e.submit_recordbatch(np.frombuffer(data, dtype=np.uint8))
        ix, space = e.rb_index(), e.rb_bytes()
        assert n == len(flat) and ix["bad"].sum() == 0
        for i, k in enumerate(flat):
            assert space[int(ix["val_off"][i]):int(ix["val_off"][i]) + int(ix["val_len"][i])].tobytes() == k.value
            assert (ix["key_len"][i] == -1) == (k.key is None)
            if k.key is not None:
                assert space[int(ix["key_off"][i]):int(ix["key_off"][i]) + int(ix["key_len"][i])].tobytes() == k.key
            assert space[int(ix["corr_off"][i]):int(ix["corr_off"][i]) + int(ix["corr_len"][i])].tobytes() == dict(k.headers)["correlation_id"]
    # the consume path replaced the plan: restore it for the tests after this one
    from calfkit import synth
    recs = synth.tool_events(3000, seed=81) + synth.tool_events(200, seed=82, size=None, full_history=True)
    b = synth.pack(recs)
    e.submit(b.data, b.offsets)
    e.tool_plan()
    e.fetch()


def test_two_calls_give_identical_bytes(planned):
    e, groups, _want = planned
    for codec in CODECS:
        for lim in (16384, 1 << 20):
            a = _encode(e, groups, compression_type=codec, max_batch_size=lim)
            b = _encode(e, groups, compression_type=codec, max_batch_size=lim)
            assert a[0] == b[0] and (a[1] == b[1]).all() and (a[2] == b[2]).all()


def test_incompressible_payloads():
    """a host tool returning ~150 KB of random text: every LZ4 frame has raw blocks (the 64 KB chunks that hold random
    text only), and both codecs stay within the stated worst case"""
    import encode_check
    import kafka_codecs as kc
    from calfkit import synth
    e = _engine(max_records=256)
    try:
        e.set_tool_node("tool.get_weather.output", None)
        recs = synth.tool_events(40, seed=83)
        b = synth.pack(recs)
        e.submit(b.data, b.offsets)
        rng = random.Random(84)
        alphabet = "abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ0123456789 .,;:-_!?"
        results = [('"' + "".join(rng.choice(alphabet) for _ in range(150000)) + '"').encode() for _ in range(e.n)]
        aux_off = np.zeros(e.n + 1, dtype=np.int64)
        np.cumsum([len(r) for r in results], out=aux_off[1:])
        e.tool_plan(np.frombuffer(b"".join(results), dtype=np.uint8), aux_off)
        out = e.fetch()
        idx = np.nonzero((out.pubs["payload"] != 0xFFFFFFFF) & (out.pubs["topic_id"] == e.topic_ids["tool.get_weather.output"]))[0]
        assert len(idx) == 40
        for codec in ("gzip", "lz4"):
            for lim in (16384, 1 << 20):
                data, off, _grp = e.encode_recordbatches(idx, timestamp_ms=TS, compression_type=codec, max_batch_size=lim)
                data = data.tobytes()
                for f in _frames(data, off):
                    plain = kc.decompress_section(CODECS[codec], f[61:])
                    assert len(f) - 61 <= len(plain) + OVERHEAD[codec](len(plain))
                    if codec == "lz4":
                        assert any(raw for raw, _n in encode_check.lz4_blocks(f[61:]))
                n = e.submit_recordbatch(np.frombuffer(data, dtype=np.uint8))
                assert n == 40 and e.rb_index()["bad"].sum() == 0
                e.submit(b.data, b.offsets)
                e.tool_plan(np.frombuffer(b"".join(results), dtype=np.uint8), aux_off)
                out = e.fetch()
    finally:
        e.close()


@pytest.mark.parametrize("limit", [16384, 1 << 20])
def test_compression_ratio_against_host_compressors(limit):
    """config-2 tool-node publishes: device gzip within 1.15 x zlib level 1, device LZ4 within 1.15 x the restated greedy
    encoder, on the same ~4 MB of sections"""
    import kafka_codecs as kc
    from calfkit import synth
    from calfkit.engine import ToolTemplate
    e = _engine(max_records=1 << 14)
    try:
        e.set_tool_node("tool.get_weather.output", ToolTemplate.from_format("It's sunny in {location}"))
        recs = synth.tool_events(1 << 14, seed=85)
        b = synth.pack(recs)
        e.submit(b.data, b.offsets)
        e.tool_plan()
        out = e.fetch()
        tid = e.topic_ids["weather_agent.input"]
        live = (out.pubs["payload"] != 0xFFFFFFFF) & (out.pubs["topic_id"] == tid)
        groups = [np.nonzero(live & (out.pubs["partition"] == p))[0] for p in range(8)]
        idx = np.concatenate(groups).astype(np.uint32)
        runs = {c: e.encode_recordbatches(idx, group_sizes=[len(g) for g in groups], timestamp_ms=TS, compression_type=c,
                                          max_batch_size=limit) for c in CODECS}
        plain = _frames(runs[None][0].tobytes(), runs[None][1])
        pick, total = [], 0
        for i in range(0, len(plain), max(1, len(plain) // 64)):
            if total >= 4 << 20:
                break
            pick.append(i)
            total += len(plain[i])
        assert total >= 1 << 20
        secs = [plain[i][61:] for i in pick]
        gz = [_frames(runs["gzip"][0].tobytes(), runs["gzip"][1])[i] for i in pick]
        lz = [_frames(runs["lz4"][0].tobytes(), runs["lz4"][1])[i] for i in pick]
        zl = sum(len(kc.gzip_encode(s, level=1)) for s in secs)
        rl = sum(len(kc.lz4_frame_encode(s, content_checksum=False)) for s in secs)
        dg, dl = sum(len(f) - 61 for f in gz), sum(len(f) - 61 for f in lz)
        assert dg <= 1.15 * zl, (dg, zl)
        assert dl <= 1.15 * rl, (dl, rl)
    finally:
        e.close()


def test_errors(planned):
    import ctypes as C
    from calfkit.engine._lib import ptr
    from calfkit.exceptions import EngineError
    e, groups, _want = planned
    g = groups[0]
    for bad in ("snappy", "zstd", "brotli", 1):
        with pytest.raises(ValueError, match="gzip"):
            e.encode_recordbatches(g, compression_type=bad)
    with pytest.raises(ValueError):
        e.encode_recordbatches(g, max_batch_size=61)
    with pytest.raises(ValueError):
        e.encode_recordbatches(g, group_sizes=[len(g) - 1])
    with pytest.raises(ValueError):
        e.encode_recordbatches(g, group_sizes=[len(g) + 1, -1])
    with pytest.raises(EngineError):                              # outside the publish table
        e.encode_recordbatches(np.array([1 << 30], dtype=np.uint32))
    # a host buffer too small: nothing is written
    idx = np.ascontiguousarray(g, dtype=np.uint32)
    goff = np.array([0, len(idx)], dtype=np.uint32)
    nf, tot = C.c_uint32(0), C.c_uint64(0)
    assert e.lib.ck_encode_recordbatches(e.h, ptr(idx), len(idx), ptr(goff), 1, None, 0, 1, 16384, C.byref(nf), C.byref(tot)) == 0
    buf = np.full(tot.value, 0xAB, dtype=np.uint8)
    with pytest.raises(EngineError, match="too small"):
        e._check(e.lib.ck_fetch_recordbatches(e.h, ptr(buf), tot.value - 1, None, None))
    assert (buf == 0xAB).all()


def test_scratch_too_small():
    """the same 100 KB publish repeated beyond what max_out / max_payloads size the scratch for: an EngineError naming the
    sizes, and the engine still encodes afterwards"""
    from calfkit import synth
    from calfkit.exceptions import EngineError
    e = _engine(max_records=64, max_in=1 << 20)
    try:
        e.set_tool_node("tool.get_weather.output", None)
        b = synth.pack(synth.tool_events(8, seed=87))
        e.submit(b.data, b.offsets)
        res = [b'"' + b"x" * 100000 + b'"'] * e.n
        aux_off = np.zeros(e.n + 1, dtype=np.int64)
        np.cumsum([len(r) for r in res], out=aux_off[1:])
        e.tool_plan(np.frombuffer(b"".join(res), dtype=np.uint8), aux_off)
        out = e.fetch(with_columns=False)
        live = np.nonzero(out.pubs["payload"] != 0xFFFFFFFF)[0]
        rep = np.full(2 * e.max_payloads, live[0], dtype=np.uint32)
        with pytest.raises(EngineError, match="exceed the scratch"):
            e.encode_recordbatches(rep, compression_type="lz4")
        data, off, _grp = e.encode_recordbatches(live, compression_type="lz4")
        assert len(off) >= 2 and off[-1] == len(data)
    finally:
        e.close()


def test_scale_one_mebi_publishes():
    """1 Mi publishes in 16 partition groups at both limits and all codecs, read back by submit_recordbatch in pieces
    under max_in_bytes"""
    from calfkit import synth
    from calfkit.engine import ToolTemplate
    n = 1 << 20
    recs = synth.tool_events(n, seed=86)
    b = synth.pack(recs)
    del recs
    e = _engine(max_records=n, max_in=int(b.data.nbytes) + (64 << 20), partitions=16)
    try:
        e.set_tool_node("tool.get_weather.output", ToolTemplate.from_format("It's sunny in {location}"))
        e.submit(b.data, b.offsets)
        e.tool_plan()
        out = e.fetch(with_columns=False)
        tid = e.topic_ids["weather_agent.input"]
        live = (out.pubs["payload"] != 0xFFFFFFFF) & (out.pubs["topic_id"] == tid)
        groups = [np.nonzero(live & (out.pubs["partition"] == p))[0] for p in range(16)]
        idx = np.concatenate(groups).astype(np.uint32)
        assert len(idx) == n
        want_len = out.out_len[out.pubs["payload"][idx]].astype(np.int64)
        sample = np.arange(0, n, 997)
        want_val = [out.payload(int(out.pubs["payload"][idx[i]])) for i in sample]
        for c in CODECS:
            for lim in (16384, 1 << 20):
                e.submit(b.data, b.offsets)                    # the read-back below replaced the plan
                e.tool_plan()
                data, off, grp = e.encode_recordbatches(idx, group_sizes=[len(g) for g in groups], timestamp_ms=TS,
                                                        compression_type=c, max_batch_size=lim)
                assert (np.diff(grp.astype(np.int64)) >= 0).all() and len(set(grp.tolist())) == 16
                lens, vals = [], {}
                piece_cap = e.max_in // (2 if c is None else 16)   # decompressed sections land in the same buffer
                i, seen = 0, 0
                while i < len(off) - 1:
                    j = i + 1
                    while j < len(off) - 1 and off[j + 1] - off[i] <= piece_cap:
                        j += 1
                    k = e.submit_recordbatch(data[off[i]:off[j]])
                    ix, space = e.rb_index(), e.rb_bytes()
                    assert ix["bad"].sum() == 0, (c, lim)
                    lens.append(ix["val_len"].astype(np.int64))
                    for s in sample[(sample >= seen) & (sample < seen + k)]:
                        o, ln = int(ix["val_off"][s - seen]), int(ix["val_len"][s - seen])
                        vals[int(s)] = space[o:o + ln].tobytes()
                    seen += k
                    i = j
                assert seen == n and (np.concatenate(lens) == want_len).all(), (c, lim)
                assert [vals[int(s)] for s in sample] == want_val, (c, lim)
    finally:
        e.close()
