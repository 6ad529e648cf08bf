"""Compressed Kafka fetches on the device: what gzip / LZ4 record batches cost against the same records uncompressed.

    python scripts/bench_kafka_codecs.py [--records 1048576] [--iters 5] [--out profiles/r03_kafka_codecs.json]

Records: config-2 tool events (synth.tool_events), about 1.1 KB each, packed into frames of 16 KB (aiokafka's default
batch size) and of 1 MB, each uncompressed, gzip level 1, gzip level 6 and LZ4 (frame defaults: independent 64 KB blocks,
content checksum).  About 64 Ki records of frames are built once and tiled to --records (baseOffset rewritten on the
copies; the CRC does not cover it).  Per case, after warm-up (inputs larger than L2):
  * compressed bytes, decompressed bytes, ratio
  * device ms per fetch from the per-kernel CUDA-event timers: "codec" = size pass + decompress, "walk" = CRC32C + split +
    field decode + the record walk, "scan" = the slot scan
  * decompressed GB/s of the codec kernels
  * end-to-end events/s from pinned host memory: submit_recordbatch + tool_plan + fetch of the payloads and publishes
  * the card's name and power limit, read in the same run
"""
from __future__ import annotations

import argparse
import json
import os
import struct
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "calfkit-sdk_b200"), ROOT, os.path.join(ROOT, "tests", "golden")):
    if p not in sys.path:
        sys.path.insert(0, p)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402

import kafka_codecs as kc  # noqa: E402
from oracle import kafka_batch as kb  # noqa: E402

TILE = 65536


def frames_of(krecs, frame_bytes: int, compression: str | None, level: int, lz4lib) -> list[bytes]:
    out, chunk, size = [], [], 0

    def flush():
        if compression == "lz4" and lz4lib is not None:
            sec = kc.liblz4_compress(lz4lib, kc.records_section(chunk), 4, False, False, False, True)
            out.append(kc.frame_with_section(sec, kc.LZ4, len(chunk)))
        elif compression == "gzip":
            out.append(kc.encode_batch(chunk, compression="gzip", level=level))
        else:
            out.append(kc.encode_batch(chunk, compression=compression))

    for k in krecs:
        if chunk and size + len(k.value) + 120 > frame_bytes:
            flush()
            chunk, size = [], 0
        chunk.append(k)
        size += len(k.value) + 120
    if chunk:
        flush()
    return out


def tile(frames: list[bytes], per_tile: int, n_records: int) -> tuple[bytes, int]:
    reps = max(1, n_records // per_tile)
    buf = bytearray()
    for t in range(reps):
        for f in frames:
            g = bytearray(f)
            struct.pack_into(">q", g, 0, t * per_tile)
            buf += g
    return bytes(buf), reps * per_tile


def card() -> dict:
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except Exception as e:  # noqa: BLE001
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def run_case(eng, buf: np.ndarray, iters: int, pinned_out: np.ndarray) -> dict:
    n = eng.submit_recordbatch(buf)                                          # warm-up
    assert eng.rb_index()["bad"].sum() == 0
    dlen = len(eng.rb_decompressed())
    eng.tool_plan(); eng._fetch(out_buf=pinned_out)
    eng.sync()
    eng.profile(True)
    eng.profile_read(reset=True)
    for _ in range(iters):
        eng.submit_recordbatch(buf)
    eng.sync()
    prof = eng.profile_read(reset=True)
    eng.profile(False)
    dev = {k: round(ms / iters, 4) for k, (ms, c) in prof.items() if c}
    t0 = time.perf_counter()
    for _ in range(iters):
        eng.submit_recordbatch(buf)
        eng.tool_plan()
        eng._fetch(out_buf=pinned_out)
    eng.sync()
    e2e = (time.perf_counter() - t0) / iters
    codec_ms = dev.get("codec", 0.0)
    return {"records": n, "fetch_bytes": int(buf.nbytes), "decompressed_bytes": dlen,
            "device_ms_per_fetch": dev,
            "codec_decompressed_GBps": round(dlen / (codec_ms * 1e-3) / 1e9, 2) if codec_ms else None,
            "e2e_ms_per_fetch": round(e2e * 1e3, 3), "e2e_events_per_s": round(n / e2e)}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=1 << 20)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_kafka_codecs.json"))
    a = ap.parse_args()
    import torch
    from calfkit import synth
    from calfkit.engine import BatchEngine, ToolTemplate
    lz4lib = kc.liblz4()
    recs = synth.tool_events(TILE, seed=2026)
    krecs = [kb.calfkit_record(r, json.loads(r)["context"]["deps"]["correlation_id"], keyed=i % 4 != 0) for i, r in enumerate(recs)]
    plain_per_tile = sum(len(kb.encode_record(k, 0, 0)) for k in krecs)
    cases = []
    eng = BatchEngine(0, max_records=a.records + 1024, max_in_bytes=int(plain_per_tile * (a.records / TILE) * 1.25) + (64 << 20))
    try:
        eng.register_topics(["tool.get_weather.input", "tool.get_weather.output", "weather_agent.input"], num_partitions=8)
        eng.set_tool_node("tool.get_weather.output", ToolTemplate.from_format("It's sunny in {location}"))
        pinned_out = torch.empty(eng.max_out + 4096, dtype=torch.uint8, pin_memory=True).numpy()
        for frame_bytes in (16 << 10, 1 << 20):
            for name, comp, level in (("none", None, 0), ("gzip-1", "gzip", 1), ("gzip-6", "gzip", 6), ("lz4", "lz4", 0)):
                frames = frames_of(krecs, frame_bytes, comp, level, lz4lib)
                raw, n = tile(frames, TILE, a.records)
                pinned = torch.empty(len(raw), dtype=torch.uint8, pin_memory=True).numpy()
                pinned[:] = np.frombuffer(raw, dtype=np.uint8)
                r = run_case(eng, pinned, a.iters, pinned_out)
                r.update({"frame_bytes": frame_bytes, "codec": name, "frames": len(frames) * (n // TILE),
                          "ratio": round(r["decompressed_bytes"] / max(1, r["fetch_bytes"] - 61 * len(frames) * (n // TILE)), 2) if comp else 1.0,
                          "lz4_encoder": ("liblz4 " + str(lz4lib.LZ4_versionNumber())) if (comp == "lz4" and lz4lib) else ("restated" if comp == "lz4" else None)})
                cases.append(r)
                print(json.dumps(r), flush=True)
                del pinned
    finally:
        eng.close()
    out = {"script": "scripts/bench_kafka_codecs.py", "records": a.records, "iters": a.iters, "card": card(), "cases": cases}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps({k: v for k, v in out.items() if k != "cases"})[:-1] + ', "cases": [\n')
        f.write(",\n".join(json.dumps(c) for c in cases) + "]}\n")


if __name__ == "__main__":
    main()
