"""CPU tests of bench.py's contract: the reference arm (`--impl reference`, the one leg that runs without a GPU) prints ONE JSON
line with the keys the driver reads, for the default config and for a sharded launch (rank 0 prints, the other ranks exit 0); and
the helpers that shape the line of the GPU arm (hypothesis ranges per rank, clock-sampler parsing) behave."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libs4ref.so")
PORT_SO = os.path.join(ROOT, "oracle", "_build", "liblcp_oracle.so")

needs_checker = pytest.mark.skipif(not (os.path.exists(REF_SO) or os.path.exists(PORT_SO)), reason="no CPU checker built (python -c 'import __graft_entry__ as g; g.build()')")

KEYS = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
        "cpu_baseline", "e2e"}


def _one_json_line(out: str) -> dict:
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


@needs_checker
@pytest.mark.timeout(300)
def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = _one_json_line(r.stdout)
    assert KEYS <= set(d), KEYS - set(d)
    assert d["impl"] == "reference" and d["unit"] == "hyp/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["n_gpus"] == 1
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


@needs_checker
@pytest.mark.timeout(300)
def test_reference_arm_under_a_two_rank_launch():
    """The driver launches the reference arm like the GPU arm (torchrun): rank 0 alone works and prints, rank 1 exits 0 silently."""
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29547",
                        os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"], capture_output=True, text=True, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    d = _one_json_line(r.stdout)
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["value"] > 0


def test_hypothesis_ranges_tile_the_global_list():
    """make_hypotheses_range (what every rank of a sharded run builds its shard with): any split reproduces the same global list."""
    sys.path.insert(0, ROOT)
    from physimglobalpose_b200 import synth
    prob = synth.make_problem(200, 2000, 0.01, seed=3)
    whole = synth.make_hypotheses_range(prob, 0, 3000, seed=9, block=1024)
    parts = [synth.make_hypotheses_range(prob, lo, hi, seed=9, block=1024) for lo, hi in ((0, 700), (700, 700), (700, 2049), (2049, 3000))]
    assert np.array_equal(np.concatenate(parts), whole)
    assert not np.array_equal(whole[:1024], whole[1024:2048])          # blocks are drawn with their own generators


def test_dumped_outputs_are_float_seeded_and_bounded(tmp_path):
    """--dump-outputs: every array is float32 / float64, a batch beyond DUMP_MAX_HYP is the same seeded sample on every call (split
    over the ranks), indices are global, and the top-k keeps its records' shape."""
    sys.path.insert(0, ROOT)
    import bench
    from physimglobalpose_b200.engine import HYP_DTYPE
    n = bench.DUMP_MAX_HYP + 4321
    counts = (np.arange(n, dtype=np.int64) * 7919 % 2001).astype(np.int32)
    scores = counts.astype(np.float32) / np.float32(2000)
    a, b = (bench.hypothesis_arrays(counts, scores, 1000, 2) for _ in range(2))
    assert len(a["counts"]) == bench.DUMP_MAX_HYP // 2 and all(np.array_equal(a[k], b[k]) for k in a)
    idx = a["hypothesis_index"].astype(np.int64) - 1000
    assert np.all(np.diff(idx) > 0) and np.array_equal(a["counts"], counts[idx]) and np.array_equal(a["scores"], scores[idx])
    small = bench.hypothesis_arrays(counts[:500], scores[:500], 0, 1)
    assert np.array_equal(small["hypothesis_index"], np.arange(500))
    top = np.zeros((4, 64), HYP_DTYPE)
    top["index"], top["T"] = np.arange(256).reshape(4, 64), 1.5
    t = bench.topk_arrays(top)
    assert t["topk_T"].shape == (4, 64, 3, 4) and np.array_equal(t["topk_index"], np.arange(256).reshape(4, 64))
    bench.dump_outputs(str(tmp_path / "out"), dict(a, **t))
    total = 0
    for name in list(a) + list(t):
        arr = np.load(tmp_path / "out" / f"{name}.npy")
        assert arr.dtype in (np.float32, np.float64)
        total += arr.nbytes
    assert total <= 64 << 20


def test_clock_sampler_parses_nvidia_smi_rows(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    s = bench.ClockSampler.__new__(bench.ClockSampler)

    class _P:
        def terminate(self): pass
        def wait(self, timeout=None): return 0
        def kill(self): pass
        def poll(self): return 0
    f = open(tmp_path / "smi.csv", "w+")
    f.write("1965, 1965, 512.3, Not Active, Not Active, Not Active, Active\n1950, 1965, 600.0, Not Active, Not Active, Not Active, Not Active\n[N/A], x\n")
    f.flush()
    s.f, s.p = f, _P()
    out = s.stop()
    assert out["sm_mhz"] == 1957.5 and out["sm_max_mhz"] == 1965 and out["reasons"] == ["sw_power_cap"] and out["samples"] == 2
