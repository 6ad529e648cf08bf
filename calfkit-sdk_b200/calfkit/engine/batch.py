"""BatchEngine: the host side of one CUDA stream's worth of the hot path.

One engine = one `ck_handle` (device buffers + stream).  It replaces, batch-wise, the reference's
per-record sandwich  bytes-in -> Envelope -> handler -> _publish_action -> bytes-out
(reference calfkit/nodes/base.py:149-164, calfkit/worker/worker.py:45-53) for the node kinds the
reference ships (@agent_tool nodes, Agent fan-out).  All decoding, routing and encoding happens in
the CUDA kernels behind the C-ABI; this class only moves buffers and interprets result tables.
"""
from __future__ import annotations

import ctypes as C
import json
import os
import string
from dataclasses import dataclass
from typing import Iterator, Sequence

import numpy as np

from calfkit.engine import _lib
from calfkit.engine._lib import COL, NUM_COLS, PUB_DTYPE, ptr
from calfkit.exceptions import EngineError


@dataclass
class ToolTemplate:
    """A tool whose return value is a pure string template of its string arguments, e.g. the
    quickstart's get_weather: f"It's sunny in {location}" (reference
    examples/quickstart/weather_tool.py:9-12).  Such tools are evaluated on the device: the JSON
    return value is assembled from pre-escaped literal pieces and the raw (already canonically
    escaped) argument strings, so no host round trip is needed.  Anything else stays a host tool."""
    kinds: list[int]          # 0 literal, 1 argument
    pieces: list[bytes]       # literal bytes (JSON-escaped) or the argument's key name

    @classmethod
    def from_format(cls, fmt: str) -> "ToolTemplate":
        kinds, pieces = [], []
        parsed = list(string.Formatter().parse(fmt))
        lit_acc = '"'
        for literal, field, spec, conv in parsed:
            lit_acc += json.dumps(literal, ensure_ascii=False)[1:-1]
            if field is not None:
                if spec or conv or not field.isidentifier():
                    raise ValueError(f"unsupported template field {field!r}")
                kinds.append(0); pieces.append(lit_acc.encode()); lit_acc = ""
                kinds.append(1); pieces.append(json.dumps(field, ensure_ascii=False)[1:-1].encode())
        lit_acc += '"'
        kinds.append(0); pieces.append(lit_acc.encode())
        return cls(kinds, pieces)


@dataclass
class Publish:
    topic: str
    key: bytes | None
    payload: bytes
    record: int
    partition: int


class _SpanOffsets:
    """offsets[i], offsets[i+1] of records that do NOT lie back to back (values inside raw Kafka frames): indexing i gives
    the start, and BatchOutput takes the end from `end(i)`"""
    def __init__(self, off: np.ndarray, ln: np.ndarray):
        self.off, self.ln = off, ln

    def __getitem__(self, i):
        return self.off[i]

    def end(self, i):
        return int(self.off[i]) + int(self.ln[i])

    def __len__(self):
        return len(self.off) + 1


class _RecordBatchBytes:
    """The byte space the offsets of `BatchEngine.rb_index()` index: the submitted buffer, followed at `base` by the
    decompressed records sections of its gzip / LZ4 frames.  Those sections are copied from the device once, on the
    first read that lands in them; a fetch whose host side reads only uncompressed records never copies them."""
    def __init__(self, engine: "BatchEngine", buf: np.ndarray, base: int):
        self.engine, self.buf, self.base = engine, buf, base
        self._submit_no = engine._submit_no
        self._dec: np.ndarray | None = None

    def decompressed(self) -> np.ndarray:
        if self._dec is None:
            if self.engine._submit_no != self._submit_no:
                raise EngineError("the decompressed records of this fetch were overwritten by a later submit: "
                                  "read them before submitting the next batch")
            self._dec = self.engine.rb_decompressed()
        return self._dec

    def __getitem__(self, s: slice) -> np.ndarray:
        start, stop = int(s.start), int(s.stop)
        if stop <= len(self.buf):
            return self.buf[start:stop]
        if start >= self.base:
            return self.decompressed()[start - self.base:stop - self.base]
        raise IndexError(f"span [{start}, {stop}) straddles the submitted and the decompressed bytes")


class BatchOutput:
    """Result of one plan+emit: unique payloads + the publish table that references them."""

    def __init__(self, engine: "BatchEngine", out: np.ndarray, out_off: np.ndarray, out_len: np.ndarray, pubs: np.ndarray,
                 in_data: np.ndarray | None, in_off: np.ndarray | None, cols: np.ndarray | None, overlay=None):
        self.engine, self.out, self.out_off, self.out_len, self.pubs = engine, out, out_off, out_len, pubs
        self.in_data, self.in_off, self.cols = in_data, in_off, cols
        self.overlay = overlay          # (bytes, off[n], len[n]): canonical re-emissions of non-canonical inputs

    def record_bytes(self, r: int) -> np.ndarray:
        """the bytes the column spans of record r refer to: its canonical re-emission if it has one"""
        if self.overlay is not None and self.overlay[1][r] >= 0:
            o = int(self.overlay[1][r])
            return self.overlay[0][o:o + int(self.overlay[2][r])]
        if isinstance(self.in_off, _SpanOffsets):
            return self.in_data[int(self.in_off[r]):self.in_off.end(r)]
        return self.in_data[self.in_off[r]:self.in_off[r + 1]]

    def payload(self, i: int) -> bytes:
        return self.out[self.out_off[i]:self.out_off[i] + self.out_len[i]].tobytes()

    def live(self) -> np.ndarray:
        return self.pubs[self.pubs["payload"] != 0xFFFFFFFF]

    def topic_of(self, p) -> str:
        if p["topic_id"] >= 0:
            return self.engine.topic_names[int(p["topic_id"])]
        rec = self.record_bytes(int(p["record"]))
        raw = rec[int(p["topic_off"]):int(p["topic_off"]) + int(p["topic_len"])].tobytes()
        return json.loads(b'"' + raw + b'"')

    def key_of(self, p) -> bytes | None:
        if not p["has_key"]:
            return None
        r = int(p["record"])
        o = int(self.cols[COL["CORR_OFF"], r])
        raw = self.record_bytes(r)[o:o + int(self.cols[COL["CORR_LEN"], r])].tobytes()
        return json.loads(b'"' + raw + b'"').encode()

    def publishes(self) -> Iterator[Publish]:
        for p in self.live():
            yield Publish(self.topic_of(p), self.key_of(p), self.payload(int(p["payload"])), int(p["record"]),
                          int(p["partition"]))


_M64 = (1 << 64) - 1


def _splitmix64(x: int) -> int:
    x = (x + 0x9E3779B97F4A7C15) & _M64
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & _M64
    return x ^ (x >> 31)


def device_uuid7_hex(unix_ms: int, seed: int, index: int) -> str:
    """The frame id the fan-out kernel writes for payload slot `index` (csrc/ck_kernels.cuh
    ck_uuid7_hex) — exposed so parity tests can inject the same ids into the oracle."""
    r0, r1 = _splitmix64((seed + 2 * index) & _M64), _splitmix64((seed + 2 * index + 1) & _M64)
    hi = ((unix_ms & 0xFFFFFFFFFFFF) << 16) | 0x7000 | (r0 & 0xFFF)
    lo = (0x2 << 62) | (r1 & 0x3FFFFFFFFFFFFFFF)
    return f"{hi:016x}{lo:016x}"


def bind_host_to_gpu(device: int) -> list[int] | None:
    """Pin the calling process to the CPUs NVML reports as local to `device` (same socket / NUMA node), so
    that pinned staging buffers allocated afterwards are first-touched next to the GPU's PCIe root.  With
    one worker process per GPU this keeps eight concurrent H2D/D2H streams off the inter-socket link.
    Returns the CPU list, or None when NVML is unavailable (nothing is changed then)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(vis.split(",")[device]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else device
        hnd = pynvml.nvmlDeviceGetHandleByIndex(idx)
        words = pynvml.nvmlDeviceGetCpuAffinity(hnd, (os.cpu_count() + 63) // 64)
        cpus = [64 * w + b for w, m in enumerate(words) for b in range(64) if (int(m) >> b) & 1]
        cpus = [c for c in cpus if c in os.sched_getaffinity(0)]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return cpus
    except Exception:
        pass
    return None


class BatchEngine:
    def __init__(self, device: int = 0, max_records: int = 1 << 16, max_in_bytes: int = 128 << 20,
                 max_out_bytes: int | None = None, max_aux_bytes: int | None = None, max_payloads: int | None = None):
        self.lib = _lib.load()
        self.max_records, self.max_in = max_records, max_in_bytes
        self.max_payloads = max_payloads if max_payloads is not None else max_records
        self.max_out = max_out_bytes if max_out_bytes is not None else max_in_bytes + 528 * max_records
        self.max_aux = max_aux_bytes if max_aux_bytes is not None else max(1 << 20, max_in_bytes // 4, 32 * self.max_payloads)
        h = C.c_void_p()
        if self.lib.ck_create(device, self.max_in, self.max_out, max_records, self.max_payloads, self.max_aux, C.byref(h)):
            raise EngineError(self.lib.ck_last_error(None).decode())
        self.h = h
        self.topic_names: dict[int, str] = {}
        self.topic_ids: dict[str, int] = {}
        self.num_partitions = 0
        self.n = 0
        self._in_data = self._in_off = None
        self._submit_no = 0                 # counts submits: the device input buffer a host view refers to is still current

    # ------------------------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "h", None):
            self.lib.ck_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int) -> None:
        if rc:
            raise EngineError(self.lib.ck_last_error(self.h).decode())

    # ------------------------------------------------------------------------------------------
    def register_topics(self, names: Sequence[str], num_partitions: int = 0) -> dict[str, int]:
        """topic string -> id table on the device (ids are positions in `names`, de-duplicated)."""
        uniq = list(dict.fromkeys(names))
        blob = b"".join(n.encode() for n in uniq)
        offs = np.zeros(len(uniq) + 1, dtype=np.uint32)
        np.cumsum([len(n.encode()) for n in uniq], out=offs[1:])
        ids = np.arange(len(uniq), dtype=np.int32)
        b = np.frombuffer(blob, dtype=np.uint8) if blob else np.zeros(1, dtype=np.uint8)
        self._check(self.lib.ck_register_topics(self.h, ptr(b), ptr(offs), len(uniq), ptr(ids), num_partitions))
        self.topic_names = dict(enumerate(uniq))
        self.topic_ids = {n: i for i, n in enumerate(uniq)}
        self.num_partitions = num_partitions
        return self.topic_ids

    def set_tool_node(self, publish_topic: str | None, template: ToolTemplate | None = None) -> None:
        pid = -1
        if publish_topic is not None:
            if publish_topic not in self.topic_ids:
                raise EngineError(f"publish topic {publish_topic!r} is not registered")
            pid = self.topic_ids[publish_topic]
        if template is None:
            self._check(self.lib.ck_set_tool_node(self.h, pid, 0, None, None, None))
            return
        kinds = np.asarray(template.kinds, dtype=np.uint32)
        blob = np.frombuffer(b"".join(template.pieces) or b"\0", dtype=np.uint8)
        offs = np.zeros(len(template.pieces) + 1, dtype=np.uint32)
        np.cumsum([len(p) for p in template.pieces], out=offs[1:])
        self._check(self.lib.ck_set_tool_node(self.h, pid, len(kinds), ptr(kinds), ptr(blob), ptr(offs)))

    def set_agent_node(self, agent_name: str, callback_topic: str, publish_topic: str | None,
                       registry: dict[str, str]) -> None:
        """registry: tool_name -> the tool node's subscribe_topics[0] (reference nodes/agent.py:71-75)."""
        missing = [t for t in list(registry.values()) + ([publish_topic] if publish_topic else []) if t not in self.topic_ids]
        if missing:
            raise EngineError(f"topics not registered: {missing}")
        esc = lambda s: json.dumps(s, ensure_ascii=False)[1:-1].encode()   # noqa: E731  spliced inside JSON strings
        names = [esc(k) for k in registry]
        topics = [esc(v) for v in registry.values()]
        nb = np.frombuffer(b"".join(names) or b"\0", dtype=np.uint8)
        tb = np.frombuffer(b"".join(topics) or b"\0", dtype=np.uint8)
        no = np.zeros(len(names) + 1, dtype=np.uint32); np.cumsum([len(x) for x in names], out=no[1:])
        to = np.zeros(len(topics) + 1, dtype=np.uint32); np.cumsum([len(x) for x in topics], out=to[1:])
        an, cb = esc(agent_name), esc(callback_topic)
        anb, cbb = np.frombuffer(an, dtype=np.uint8), np.frombuffer(cb, dtype=np.uint8)
        pid = self.topic_ids[publish_topic] if publish_topic else -1
        self._check(self.lib.ck_set_agent_node(self.h, pid, ptr(anb), len(an), ptr(cbb), len(cb), ptr(nb), ptr(no),
                                               ptr(tb), ptr(to), len(names)))
        ids = np.asarray([self.topic_ids[v] for v in registry.values()] or [0], dtype=np.uint32)
        self._check(self.lib.ck_set_agent_tool_topic_ids(self.h, self.topic_ids.get(callback_topic, -1), ptr(ids), len(registry)))

    def fanout_plan(self, unix_ms: int, seed: int, max_fanout: int = 128, sequential: bool = False) -> None:
        """list[Call] / Call of the pending tool calls; sequential: first pending only (agent.py:94-108)."""
        self._check(self.lib.ck_fanout_plan(self.h, unix_ms, seed, max_fanout, 1 if sequential else 0))

    def tailcall_plan(self, unix_ms: int, seed: int) -> None:
        """TailCall to the agent's own subscribe topic (agent.py:171-175)."""
        self._check(self.lib.ck_tailcall_plan(self.h, unix_ms, seed))

    def set_bucketing(self, on: bool = True) -> None:
        """bucket every submitted batch by record length before the walk (topics with mixed record sizes / shapes)"""
        self._check(self.lib.ck_set_option(self.h, 1, 1 if on else 0))

    # ---- aggregation gate on the device (csrc/ck_gate.cuh; reference nodes/agent.py:57-68) ---------------------------
    def gate_create(self, max_entries: int = 1 << 14, max_slots: int | None = None, arena_bytes: int = 256 << 20) -> None:
        self._check(self.lib.ck_gate_create(self.h, max_entries, max_slots if max_slots is not None else 16 * max_entries, arena_bytes))
        self.gate_arena_bytes = arena_bytes

    def gate_register(self, min_pending: int = 2) -> None:
        """after fanout_plan: every record that went out as list[Call] becomes a pending entry of the gate"""
        self._check(self.lib.ck_gate_register(self.h, min_pending))

    def gate_arrive(self, stamp_base: int) -> None:
        """run the gate over the submitted batch of arrivals; ACTION afterwards: SILENT / GATE_COMPLETE / GATE_PASS"""
        self._check(self.lib.ck_gate_arrive(self.h, stamp_base))

    def gate_stats(self) -> dict[str, int]:
        out = np.zeros(5, dtype=np.uint64)
        self._check(self.lib.ck_gate_stats(self.h, ptr(out)))
        st = dict(zip(["entries_used", "slots_used", "arena_used", "live", "failures"], (int(x) for x in out)))
        if st["failures"]:
            raise EngineError(f"aggregation gate out of capacity ({st}): raise max_entries / max_slots / arena_bytes")
        return st

    def gate_reset(self) -> None:
        self._check(self.lib.ck_gate_reset(self.h))

    # ------------------------------------------------------------------------------------------
    def submit(self, data: np.ndarray, offsets: np.ndarray) -> None:
        """H2D + decode of a host batch (uint8 bytes, int64 offsets[n+1]); asynchronous."""
        assert data.dtype == np.uint8 and offsets.dtype == np.int64
        self.n = len(offsets) - 1
        self._submit_no += 1
        self._in_data, self._in_off = data, offsets
        self._check(self.lib.ck_submit(self.h, ptr(data), ptr(offsets), self.n))

    def submit_recordbatch(self, buf: np.ndarray) -> int:
        """H2D + CRC32C check + record split + field decode + walk of a fetch response's record set (concatenated Kafka
        RecordBatch v2 frames, uncompressed or compressed with gzip / LZ4, which are decompressed on the device); returns
        the number of records.  Column spans are relative to each VALUE.  Raises EngineError if the submitted plus the
        decompressed bytes exceed max_in_bytes."""
        assert buf.dtype == np.uint8
        n = C.c_uint32(0)
        self._submit_no += 1
        self._check(self.lib.ck_submit_recordbatch(self.h, ptr(buf), buf.nbytes, C.byref(n)))
        self.n = n.value
        idx = self.rb_index()
        base, length = C.c_uint64(0), C.c_uint64(0)
        self._check(self.lib.ck_fetch_rb_decompressed(self.h, None, 0, C.byref(base), C.byref(length)))
        # the host-side view of the batch for result decoding: record i = data[val_off[i] : val_off[i] + val_len[i]]
        data = _RecordBatchBytes(self, buf, base.value) if length.value else buf
        self._in_data, self._in_off = data, _SpanOffsets(idx["val_off"], idx["val_len"])
        self._rb = idx
        return self.n

    def rb_decompressed(self) -> np.ndarray:
        """the decompressed records sections of the last submit_recordbatch (one device-to-host copy); they start at
        offset `len(buf)` rounded up to 16 of the space rb_index() offsets index.  Empty if no frame was compressed."""
        base, length = C.c_uint64(0), C.c_uint64(0)
        self._check(self.lib.ck_fetch_rb_decompressed(self.h, None, 0, C.byref(base), C.byref(length)))
        out = np.empty(max(length.value, 1), dtype=np.uint8)
        if length.value:
            self._check(self.lib.ck_fetch_rb_decompressed(self.h, ptr(out), out.nbytes, C.byref(base), C.byref(length)))
        return out[:length.value]

    def rb_bytes(self) -> np.ndarray | _RecordBatchBytes:
        """the byte space rb_index() offsets index (slice it as data[start:stop]): the submitted buffer, followed by the
        decompressed records sections of its compressed frames"""
        return self._in_data

    def rb_index(self) -> dict[str, np.ndarray]:
        """where value / key / the correlation_id header of every record lie (len -1 = absent): offsets into the submitted
        buffer followed by the decompressed sections of compressed frames (see rb_bytes()).  bad: 0, or why the record's
        frame was refused — 1 CRC / framing / decompression failure, 2 a codec not decoded on the device (snappy, zstd)"""
        n = self.n
        out = {"val_off": np.zeros(n, np.int64), "val_len": np.zeros(n, np.uint32), "key_off": np.zeros(n, np.int64),
               "key_len": np.zeros(n, np.int32), "corr_off": np.zeros(n, np.int64), "corr_len": np.zeros(n, np.int32),
               "bad": np.zeros(n, np.uint32)}
        if n:
            self._check(self.lib.ck_fetch_rb_index(self.h, *[ptr(out[k]) for k in ("val_off", "val_len", "key_off", "key_len", "corr_off", "corr_len", "bad")]))
        return out

    def encode_recordbatch(self, pub_indices: np.ndarray, base_offset: int = 0, timestamp_ms: int = 0) -> np.ndarray:
        """one Kafka RecordBatch v2 frame holding the publishes `pub_indices` of the current plan (one topic-partition, in
        send order), built on the device"""
        idx = np.ascontiguousarray(pub_indices, dtype=np.uint32)
        cap = self.max_out + 256 * self.max_payloads + 4096
        buf = np.empty(cap, dtype=np.uint8)
        used = C.c_uint64(0)
        self._check(self.lib.ck_encode_recordbatch(self.h, ptr(idx), len(idx), base_offset, timestamp_ms, ptr(buf), cap, C.byref(used)))
        return buf[:used.value]

    _CODECS = {None: 0, "gzip": 1, "lz4": 3}

    def encode_recordbatches(self, pub_indices: np.ndarray, group_sizes: Sequence[int] | None = None,
                             base_offsets: Sequence[int] | None = None, timestamp_ms: int = 0,
                             compression_type: str | None = None, max_batch_size: int = 16384
                             ) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """the publishes `pub_indices` of the current plan, in groups of `group_sizes` consecutive indices (one
        topic-partition each, in send order; None = one group), as runs of Kafka RecordBatch v2 frames built on the device:
        a frame takes its group's next records while it stays within `max_batch_size` bytes (always at least one record),
        and its records section is compressed with `compression_type` (None, "gzip" or "lz4", aiokafka's names).  Frame k
        of group g starts at offset base_offsets[g] (default 0) plus the records of g in earlier frames.
        Returns (data, frame_off, frame_group): frame i = data[frame_off[i]:frame_off[i + 1]], from group frame_group[i]."""
        if compression_type not in self._CODECS:
            raise ValueError(f"compression_type {compression_type!r} is not supported: use None, 'gzip' or 'lz4'")
        if max_batch_size < 62:
            raise ValueError(f"max_batch_size {max_batch_size} is below 62 (a 61-byte header and one record byte)")
        idx = np.ascontiguousarray(pub_indices, dtype=np.uint32)
        sizes = np.asarray([len(idx)] if group_sizes is None else list(group_sizes), dtype=np.int64)
        if (sizes < 0).any() or int(sizes.sum()) != len(idx):
            raise ValueError(f"group_sizes must be non-negative and sum to len(pub_indices) = {len(idx)}")
        goff = np.zeros(len(sizes) + 1, dtype=np.uint32)
        np.cumsum(sizes, out=goff[1:])
        base = None
        if base_offsets is not None:
            base = np.ascontiguousarray(base_offsets, dtype=np.int64)
            if len(base) != len(sizes):
                raise ValueError(f"base_offsets must have one entry per group ({len(sizes)})")
        nf, total = C.c_uint32(0), C.c_uint64(0)
        self._check(self.lib.ck_encode_recordbatches(self.h, ptr(idx), len(idx), ptr(goff), len(sizes), ptr(base), timestamp_ms,
                                                     self._CODECS[compression_type], max_batch_size, C.byref(nf), C.byref(total)))
        data = np.empty(max(total.value, 1), dtype=np.uint8)
        frame_off = np.zeros(nf.value + 1, dtype=np.uint64)
        frame_group = np.zeros(max(nf.value, 1), dtype=np.uint32)
        self._check(self.lib.ck_fetch_recordbatches(self.h, ptr(data), data.nbytes, ptr(frame_off), ptr(frame_group)))
        return data[:total.value], frame_off.astype(np.int64), frame_group[:nf.value]

    def submit_device(self, dev_data, dev_off, n: int, host_data: np.ndarray | None = None,
                      host_off: np.ndarray | None = None) -> None:
        """decode a batch already resident in HBM (torch tensors or raw device addresses)."""
        self.n = n
        self._submit_no += 1
        self._in_data, self._in_off = host_data, host_off
        a = dev_data if isinstance(dev_data, int) else ptr(dev_data)
        b = dev_off if isinstance(dev_off, int) else ptr(dev_off)
        self._check(self.lib.ck_submit_device(self.h, a, b, n))

    def tool_args(self) -> tuple[np.ndarray, np.ndarray]:
        """(blob, offsets[n+1]): the `args` JSON of every record that reaches the tool (host tools)."""
        self._check(self.lib.ck_tool_args(self.h))
        out, off, ln, _ = self._fetch(want_pubs=False)
        return out, off, ln

    def tool_plan(self, aux: np.ndarray | None = None, aux_off: np.ndarray | None = None) -> None:
        self._check(self.lib.ck_tool_plan(self.h, ptr(aux), ptr(aux_off)))

    def reply_plan(self, mode: int = 0) -> None:
        """client reply decode (client/deserialize.py:55-89): payload i = output value JSON; mode 0 auto, 1 text, 2 data"""
        self._check(self.lib.ck_reply_plan(self.h, mode))

    def return_plan(self) -> None:
        self._check(self.lib.ck_return_plan(self.h))

    def tool_plan_device(self, dev_aux, dev_aux_off) -> None:
        self._check(self.lib.ck_tool_plan_device(self.h, ptr(dev_aux), ptr(dev_aux_off)))

    def launch_count(self) -> int:
        """kernels launched by this engine so far"""
        return int(self.lib.ck_launch_count(self.h))

    def sync(self) -> None:
        self._check(self.lib.ck_sync(self.h))

    def columns(self) -> np.ndarray:
        cols = np.empty((NUM_COLS, self.n), dtype=np.uint32)
        if self.n:
            self._check(self.lib.ck_fetch_columns(self.h, ptr(cols)))
        return cols

    def out_size(self) -> tuple[int, int, int]:
        nb, npay, npub = C.c_uint64(), C.c_uint32(), C.c_uint32()
        self._check(self.lib.ck_out_size(self.h, C.byref(nb), C.byref(npay), C.byref(npub)))
        return nb.value, npay.value, npub.value

    def _fetch(self, want_pubs: bool = True, out_buf: np.ndarray | None = None, off_buf: np.ndarray | None = None,
               len_buf: np.ndarray | None = None, pubs_buf: np.ndarray | None = None):
        """D2H of the results.  The optional *_buf arrays let a caller land everything in pinned memory it
        owns (required for copies that overlap with the other PCIe direction)."""
        nb, npay, npub = self.out_size()
        out = out_buf if out_buf is not None else np.empty(max(nb, 1), dtype=np.uint8)
        off = off_buf[:npay + 1] if off_buf is not None else np.zeros(npay + 1, dtype=np.int64)
        ln = len_buf[:npay] if len_buf is not None else np.zeros(npay, dtype=np.uint32)
        npub_eff = npub if want_pubs else 0
        pubs = pubs_buf[:npub_eff] if pubs_buf is not None else np.zeros(npub_eff, dtype=PUB_DTYPE)
        self._check(self.lib.ck_fetch_output(self.h, ptr(out), out.nbytes, ptr(off) if npay else None,
                                             ptr(ln) if npay else None, ptr(pubs) if npub_eff else None))
        return out[:nb], off, ln, pubs

    def fetch(self, out_buf: np.ndarray | None = None, with_columns: bool = True) -> BatchOutput:
        out, off, ln, pubs = self._fetch(out_buf=out_buf)
        cols = self.columns() if with_columns else None
        return BatchOutput(self, out, off, ln, pubs, self._in_data, self._in_off, cols, self.overlay())

    def overlay(self):
        """(bytes, off[n], len[n]) of the canonicalised records of the current batch, or None if there are none"""
        if not self.n:
            return None
        off = np.empty(self.n, dtype=np.int64)
        ln = np.empty(self.n, dtype=np.uint32)
        buf = np.empty(self.max_in + 256, dtype=np.uint8)
        used = C.c_uint64(0)
        self._check(self.lib.ck_fetch_overlay(self.h, ptr(buf), buf.nbytes, ptr(off), ptr(ln), C.byref(used)))
        if not (off >= 0).any():
            return None
        return buf[:used.value], off, ln

    # ------------------------------------------------------------------------------------------
    def stream_ptr(self) -> int:
        return int(self.lib.ck_stream(self.h))

    def device_buffers(self) -> dict[str, int]:
        ps = [C.c_void_p() for _ in range(5)]
        self._check(self.lib.ck_device_buffers(self.h, *[C.byref(p) for p in ps]))
        return dict(zip(["in", "in_off", "out", "out_off", "cols"], [p.value for p in ps]))

    def profile(self, enable: bool) -> None:
        self._check(self.lib.ck_profile(self.h, int(enable)))

    def profile_read(self, reset: bool = True) -> dict[str, tuple[float, int]]:
        ms = np.zeros(_lib.NUM_KERNELS, dtype=np.float32)
        cnt = np.zeros(_lib.NUM_KERNELS, dtype=np.uint32)
        self._check(self.lib.ck_profile_read(self.h, ptr(ms), ptr(cnt), int(reset)))
        return {k: (float(ms[i]), int(cnt[i])) for i, k in enumerate(_lib.KERNELS)}

    # ------------------------------------------------------------------------------------------
    def run_tool_batch(self, data: np.ndarray, offsets: np.ndarray, host_tool=None) -> BatchOutput:
        """Convenience: one full tool-node step over a host batch.  `host_tool(args_json: bytes) ->
        result_json: bytes` is used when the node has no device template."""
        self.submit(data, offsets)
        if host_tool is None:
            self.tool_plan()
        else:
            blob, off, ln = self.tool_args()
            results = [host_tool(blob[off[i]:off[i] + ln[i]].tobytes()) if ln[i] else b"" for i in range(self.n)]
            aux_off = np.zeros(self.n + 1, dtype=np.int64)
            np.cumsum([len(r) for r in results], out=aux_off[1:])
            aux = np.frombuffer(b"".join(results) or b"\0", dtype=np.uint8)
            self.tool_plan(aux, aux_off)
        return self.fetch()
