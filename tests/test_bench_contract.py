"""bench.py's reference arm (`--impl reference`) runs entirely on the CPU, so its JSON contract is checked here; the
product arm prints the same keys plus clocks / gpu_launches / roofline, and can dump the outputs of its timed steps."""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines                      # exactly ONE JSON line on stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "mono_equiv_samples_per_sec" and d["unit"] == "samples/s"
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["config"]["workload"].startswith("c2")    # BASELINE configs[1], the headline configuration
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


@pytest.mark.gpu
def test_dump_outputs_repeat_bit_for_bit(gpu, tmp_path):
    """--dump-outputs writes each config's last timed step; the same arguments give the same files. c3 carries filter and
    delay state across steps, and its 512 MiB of per-voice output is cut to a seeded sample of voices."""
    dumps = []
    for i in range(2):
        out = tmp_path / f"run{i}"
        r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--only", "c2,c3", "--steps", "3", "--warmup", "1", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=900, cwd=str(ROOT), env=dict(os.environ, FW_BENCH_SKIP_CPU="1"))
        assert r.returncode == 0, r.stderr[-2000:]
        d = json.loads(r.stdout.strip().splitlines()[-1])
        assert d["steps"] == 3 and d["configs"]["c3"]["timed_steps"] == 3
        assert sorted(p.name for p in out.iterdir()) == ["c2.npy", "c3.npy"]
        assert sum(p.stat().st_size for p in out.iterdir()) <= 64_000_000
        dumps.append({n: np.load(out / f"{n}.npy") for n in ("c2", "c3")})
    c2, c3 = dumps[0]["c2"], dumps[0]["c3"]
    assert c2.dtype == np.float32 and c2.shape == (2, 256 * 256)
    assert c3.dtype == np.float32 and c3.shape[1:] == (2, 32 * 512) and 0 < c3.shape[0] < 4096
    for a in (c2, c3):
        assert np.all(np.isfinite(a)) and np.abs(a).max() > 0
    for n in ("c2", "c3"):
        assert np.array_equal(dumps[0][n].view(np.uint32), dumps[1][n].view(np.uint32)), n
