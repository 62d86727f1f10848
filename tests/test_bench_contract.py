"""bench.py --impl reference on the CPU (no GPU needed): the JSON line carries the contract's keys and the arm is the
unmodified reference when oracle/_ref has been built (oracle/build_ref.py), the labelled oracle port otherwise."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", XFEAT_BENCH_CPU_PAIRS="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, env=env, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "pairs/s" and d["higher_is_better"] is True and d["n_gpus"] == 1
    assert d["steps"] == 2 and d["warmup"] == 1 and d["steps_requested"] == 2
    assert d["value"] > 0 and abs(d["ms_per_step"] - 1e3 / d["value"]) < 1e-6 * d["ms_per_step"]
    assert d["metric"].startswith("image-pairs/sec") and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert set(cb) >= {"value", "unit", "cores", "kind", "sample"} and cb["value"] == d["value"] and cb["cores"] >= 1
    from oracle import build_ref
    assert cb["kind"] == ("reference" if build_ref.available() else "port")
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_dump_outputs_are_float_and_zero_past_each_count(tmp_path):
    import numpy as np
    import torch
    import bench
    g = torch.Generator().manual_seed(0)
    mk0, mk1 = torch.rand(3, 5, 2, generator=g), torch.rand(3, 5, 2, generator=g)
    cnt = torch.tensor([2, 0, -1], dtype=torch.int32)                  # -1: the overflow status of a pair
    n = torch.tensor([5, 4, 3], dtype=torch.int32)
    want0 = mk0.numpy().copy()
    bench.write_outputs(str(tmp_path / "sparse"), bench.last_step_outputs((mk0, mk1, cnt, n, n), star=False))
    got = {p.stem: np.load(p) for p in (tmp_path / "sparse").iterdir()}
    assert set(got) == {"mkpts0", "mkpts1", "n_matches", "n_keypoints0", "n_keypoints1"}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert np.array_equal(got["mkpts0"][0, :2], want0[0, :2]) and not got["mkpts0"][0, 2:].any() and not got["mkpts0"][1:].any()
    assert got["n_matches"].tolist() == [2, 0, -1] and got["n_keypoints0"].tolist() == [5, 4, 3]
    m = torch.rand(2, 4, 4, generator=g)
    want = m.numpy().copy()
    star = bench.last_step_outputs((m, torch.tensor([4, 1], dtype=torch.int32), torch.tensor([9, 7], dtype=torch.int32)), star=True)
    assert np.array_equal(star["matches"][0], want[0]) and np.array_equal(star["matches"][1, :1], want[1, :1])
    assert not star["matches"][1, 1:].any() and star["n_coarse_matches"].tolist() == [9, 7]


def test_non_zero_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, env=env, timeout=300, cwd=ROOT)
    assert r.returncode == 0 and r.stdout.strip() == ""
