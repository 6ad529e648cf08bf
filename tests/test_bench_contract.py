"""bench.py's reference arm on CPU (the GPU arm needs a B200): one JSON line on stdout with the contract's keys."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, p.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "agent_events_per_sec" and d["unit"] == "events/s"
    for key in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype", "data", "config"):
        assert key in d
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 0


_FAKE_ENGINE = r'''
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import bench
from calfkit.engine._lib import NUM_COLS, PUB_DTYPE

class Engine:
    """the last plan of a 50 000-record batch: payload i (16-byte padded in the buffer) belongs to record i and is
    published twice; every 7th record publishes nothing"""
    def __init__(self):
        rng = np.random.default_rng(5)
        n = 50_000
        ln = rng.integers(200, 1500, size=n).astype(np.uint32)
        off = np.zeros(n + 1, np.int64)
        off[1:] = np.cumsum((ln.astype(np.int64) + 15) // 16 * 16)
        self.out = rng.integers(0, 256, size=int(off[-1]), dtype=np.uint8)
        self.off, self.ln = off, ln
        self.pubs = np.zeros(2 * n, PUB_DTYPE)
        self.pubs["payload"] = np.repeat(np.arange(n), 2)
        self.pubs["payload"][np.repeat(np.arange(n) % 7 == 0, 2)] = 0xFFFFFFFF
        self.pubs["record"] = np.repeat(np.arange(n), 2)
        self.pubs["topic_id"] = np.tile([2, 1], n)
        self.pubs["partition"] = rng.integers(0, 8, size=2 * n)
        self.cols = rng.integers(0, 1 << 20, size=(NUM_COLS, n)).astype(np.uint32)
    def _fetch(self):
        return self.out, self.off, self.ln, self.pubs
    def columns(self):
        return self.cols

bench.dump_outputs(sys.argv[2], Engine())
'''


def test_dump_outputs_float_arrays_seeded_and_bounded(tmp_path):
    """--dump-outputs: every file is a float32 / float64 .npy, the whole dump stays under 64 MB, two dumps of the same
    outputs are identical, and the sampled publishes and payloads are exactly what the engine returned"""
    import numpy as np
    script = tmp_path / "dump.py"
    script.write_text(_FAKE_ENGINE)
    dirs = [tmp_path / "a", tmp_path / "b"]
    for d in dirs:
        p = subprocess.run([sys.executable, str(script), ROOT, str(d)], capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert p.returncode == 0, p.stderr[-2000:]
    names = sorted(f.name for f in dirs[0].iterdir())
    assert names == sorted(f"{k}.npy" for k in ("totals", "records", "columns", "publishes", "payload_index", "payload_len", "payloads"))
    assert sum(f.stat().st_size for f in dirs[0].iterdir()) <= 64 << 20
    a = {f[:-4]: np.load(dirs[0] / f) for f in names}
    for f in names:
        assert a[f[:-4]].dtype in (np.float32, np.float64)
        assert np.array_equal(a[f[:-4]], np.load(dirs[1] / f))
    n = 50_000
    assert a["totals"][:3].tolist() == [n, n, 2 * (n - (n + 6) // 7)]
    assert len(a["records"]) == 4096 and a["columns"].shape[1] == 4096
    pubs = a["publishes"].astype(np.int64)
    assert len(pubs) and (pubs[:, 0] == pubs[:, 4]).all() and np.isin(pubs[:, 4], a["records"]).all()
    assert a["payloads"].size == a["payload_len"].sum() <= 8 << 20
    rng = np.random.default_rng(5)
    ln = rng.integers(200, 1500, size=n)
    off = np.concatenate([[0], np.cumsum((ln + 15) // 16 * 16)])
    out = rng.integers(0, 256, size=int(off[-1]), dtype=np.uint8)
    idx = a["payload_index"].astype(np.int64)
    assert (a["payload_len"] == ln[idx]).all()
    assert np.array_equal(a["payloads"], np.concatenate([out[off[i]:off[i] + ln[i]] for i in idx]).astype(np.float32))


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert p.returncode == 0 and p.stdout.strip() == "", (p.stdout[-500:], p.stderr[-500:])
