"""Compressed Kafka produce on the device: what encode_recordbatches costs per codec and batch size.

    python scripts/bench_kafka_produce.py [--records 1048576] [--iters 5] [--out profiles/r04_kafka_produce.json]

Setup: --records config-2 tool events (synth.tool_events, about 1.1 KB each) -> tool_plan -> the live publishes grouped
per (topic, partition) (keyed weather_agent.input publishes over 8 partitions, and the unkeyed tool.get_weather.output
publishes as one more group) -> one encode_recordbatches call per step.  Cases: no compression, gzip and LZ4, each at
max_batch_size 16384 (aiokafka's default) and 1 MiB.  Per case, after a warm-up call:
  * frames, plaintext (records section) bytes, compressed section bytes, ratio
  * device ms per call from the per-kernel CUDA-event timers: "codec" = the compression kernels, "emit" = split, record
    writes, assembly, headers and CRC32C, "scan" = the prefix sums
  * plaintext GB/s over all device time and over the codec kernels alone
  * wall ms per call including the device-to-host copy of the frames (pageable host memory)
  * one host core compressing a sample of the same sections: zlib level 1, and liblz4 (default settings) where it loads
The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "calfkit-sdk_b200"), ROOT, os.path.join(ROOT, "tests", "golden")):
    if p not in sys.path:
        sys.path.insert(0, p)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402

import kafka_codecs as kc  # noqa: E402


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


def host_rate(sections: list[bytes], lz4lib) -> dict:
    """one host core on the same sections: zlib level 1 (raw deflate + gzip framing cost is negligible) and liblz4"""
    n = sum(len(s) for s in sections)
    t0 = time.perf_counter()
    zl = sum(len(zlib.compress(s, 1)) for s in sections)
    tz = time.perf_counter() - t0
    out = {"sample_bytes": n, "zlib1_MBps": round(n / tz / 1e6, 1), "zlib1_ratio": round(n / zl, 2)}
    if lz4lib is not None:
        t0 = time.perf_counter()
        lz = sum(len(kc.liblz4_compress(lz4lib, s)) for s in sections)
        tl = time.perf_counter() - t0
        out.update({"liblz4_MBps": round(n / tl / 1e6, 1), "liblz4_ratio": round(n / lz, 2)})
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=1 << 20)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_kafka_produce.json"))
    a = ap.parse_args()
    from calfkit import synth
    from calfkit.engine import BatchEngine, ToolTemplate
    lz4lib = kc.liblz4()
    b = synth.pack(synth.tool_events(a.records, seed=1000))
    eng = BatchEngine(0, max_records=a.records, max_in_bytes=int(b.data.nbytes) + 4096)
    cases = []
    try:
        eng.register_topics(["tool.get_weather.input", "tool.get_weather.output", "weather_agent.input"], num_partitions=8)
        eng.set_tool_node("tool.get_weather.output", ToolTemplate.from_format("It's sunny in {location}"))
        eng.submit(b.data, b.offsets)
        eng.tool_plan()
        pubs = eng.fetch(with_columns=False).pubs
        live = np.nonzero(pubs["payload"] != 0xFFFFFFFF)[0]
        order = live[np.lexsort((live, pubs["partition"][live], pubs["topic_id"][live]))]   # stable: send order per group
        key = pubs["topic_id"][order].astype(np.int64) * 4096 + pubs["partition"][order]
        sizes = np.diff(np.flatnonzero(np.r_[True, key[1:] != key[:-1], True]))
        idx = order.astype(np.uint32)
        plain_by_limit = {}
        for limit in (16384, 1 << 20):
            for codec in (None, "gzip", "lz4"):
                call = lambda: eng.encode_recordbatches(idx, group_sizes=sizes, timestamp_ms=1767225600000,  # noqa: E731
                                                        compression_type=codec, max_batch_size=limit)
                data, off, _grp = call()                                           # warm-up (and scratch allocation)
                frames = len(off) - 1
                sec_bytes = int(data.nbytes) - 61 * frames
                if codec is None:
                    plain_by_limit[limit] = sec_bytes
                    step = max(1, frames // 256)
                    sample = [data[off[i] + 61:off[i + 1]].tobytes() for i in range(0, frames, step)][:64]
                eng.sync()
                eng.profile(True)
                eng.profile_read(reset=True)
                for _ in range(a.iters):
                    call()
                eng.sync()
                prof = eng.profile_read(reset=True)
                eng.profile(False)
                dev = {k: round(ms / a.iters, 4) for k, (ms, c) in prof.items() if c}
                t0 = time.perf_counter()
                for _ in range(a.iters):
                    call()
                wall = (time.perf_counter() - t0) / a.iters
                plain = plain_by_limit[limit]
                dev_ms = sum(dev.values())
                r = {"codec": codec or "none", "max_batch_size": limit, "publishes": int(len(idx)), "groups": int(len(sizes)),
                     "frames": frames, "plaintext_bytes": plain, "section_bytes": sec_bytes, "ratio": round(plain / sec_bytes, 3),
                     "device_ms_per_call": dev, "device_ms_total": round(dev_ms, 4),
                     "plaintext_GBps_device": round(plain / (dev_ms * 1e-3) / 1e9, 2) if dev_ms else None,
                     "plaintext_GBps_codec_kernels": round(plain / (dev["codec"] * 1e-3) / 1e9, 2) if dev.get("codec") else None,
                     "wall_ms_per_call_with_fetch": round(wall * 1e3, 3)}
                if codec is not None:
                    r["host_one_core"] = host_rate(sample, lz4lib)
                cases.append(r)
                print(json.dumps(r), flush=True)
    finally:
        eng.close()
    out = {"script": "scripts/bench_kafka_produce.py", "records": a.records, "iters": a.iters, "card": card(), "cases": cases}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps({k: v for k, v in out.items() if k != "cases"})[:-1] + ', "cases": [\n')
        f.write(",\n".join(json.dumps(c) for c in cases) + "]}\n")


if __name__ == "__main__":
    main()
