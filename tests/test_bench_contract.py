"""bench.py contract on the CPU: the reference arm prints one JSON line with the driver's keys; the B200 arm refuses to run
without a CUDA device (no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, env=e, timeout=600)


def test_reference_arm_prints_the_contract_line():
    r = run("--impl", "reference", "--config", "c1", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["metric"] == "reconstructed_points_per_sec" and d["unit"] == "points/s"
    assert d["steps"] == 1 and d["warmup"] == 0 and d["higher_is_better"] is True and d["value"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == 1 and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("c1")


def test_reference_arm_under_torchrun_only_rank0_prints():
    r = run("--impl", "reference", "--config", "c1", "--steps", "1", "--warmup", "0", env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_b200_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    r = run("--steps", "1", "--warmup", "0")
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_strong_scaling_plan_covers_the_sequence():
    """bench.py's N > 1 workload (BASELINE config 3, strong scaling): the ranks' GOF lists tile the 300-frame sequence exactly,
    cut at the sequence's GOF boundaries; both arms derive the same `config` dict from the same arguments."""
    import argparse
    bench = load_bench()
    for world in (1, 2, 3, 4, 8):
        sizes = [bench.rank_gofs("strong", 30, r, world) for r in range(world)]
        assert sum(sum(s) for s in sizes) == bench.SEQ_FRAMES
        assert all(0 < g <= bench.SEQ_GOF for s in sizes for g in s)
        f = 0
        for s in sizes:                                   # contiguous slices; no GOF of a rank straddles a sequence GOF boundary
            for g in s:
                assert f // bench.SEQ_GOF == (f + g - 1) // bench.SEQ_GOF
                f += g
    args = argparse.Namespace(config="auto", frames=0, no_smoothing=False, gpus=8)
    mode, sname, frames, smoothing, desc = bench.workload(args, 8)
    assert (mode, sname, frames, smoothing) == ("strong", "c3", 30, True) and desc["frames_per_step"] == 300
    assert bench.workload(args, 1) == bench.workload(args, 8)                 # --gpus 8 without torchrun (the reference arm): same dict
    args1 = argparse.Namespace(config="auto", frames=0, no_smoothing=False, gpus=1)
    mode1, sname1, frames1, _, desc1 = bench.workload(args1, 1)
    assert (mode1, sname1, frames1) == ("weak", "c2", 32) and desc1["atlas"] == "1024x1024"
    assert bench.rank_gofs("weak", 32, 0, 1) == [32] * bench.GOFS_PER_STEP


def load_bench():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


DUMP_NAMES = {"points_per_frame", "frame_sums", "sample_index", "sample_positions", "sample_colors"}


def test_dump_outputs_files_counts_sums_and_sample(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float .npy files holding every frame's point count and column sums, and a seeded sample of its
    points (the same on every run) that stays within the sample budget."""
    import numpy as np
    bench = load_bench()
    assert bench.DUMP_POINTS * 40 < 64 << 20
    monkeypatch.setattr(bench, "DUMP_POINTS", 1000)
    rng = np.random.RandomState(0)
    frames = [(rng.randint(0, 1024, (n, 3)).astype(np.uint16), rng.randint(0, 256, (n, 3)).astype(np.uint8))
              for n in (0, 7, 5000, 300000)]
    a = bench.dump_outputs(str(tmp_path / "a"), frames)
    monkeypatch.setattr(bench, "DUMP_POINTS", 2000)                          # two ranks: the same share each as above
    bench.dump_outputs(str(tmp_path / "b"), frames, rank=1, world=2)
    assert set(a) == DUMP_NAMES
    for name, arr in a.items():
        got = np.load(tmp_path / "a" / f"{name}.npy")
        assert got.dtype in (np.float32, np.float64) and np.array_equal(got, arr)
        assert np.array_equal(np.load(tmp_path / "b" / f"rank1_{name}.npy"), arr)
    assert a["points_per_frame"].tolist() == [0, 7, 5000, 300000]
    idx = a["sample_index"].astype(np.int64)
    assert len(idx) == 0 + 7 + 250 + 250 and len(np.unique(idx, axis=0)) == len(idx)
    for j, (p, c) in enumerate(frames):
        assert a["frame_sums"][j].tolist() == p.sum(0).tolist() + c.sum(0).tolist()
        rows = idx[:, 0] == j
        assert np.array_equal(a["sample_positions"][rows], p[idx[rows, 1]])
        assert np.array_equal(a["sample_colors"][rows], c[idx[rows, 1]])


@pytest.mark.parametrize("world", [1, 2, 8])
def test_dump_outputs_all_ranks_stay_within_64mb(tmp_path, world):
    """Under torchrun every rank writes its own files into the same DIR: together they stay within 64 MB."""
    import numpy as np
    bench = load_bench()
    rng = np.random.RandomState(1)
    frames = [(rng.randint(0, 1024, (n, 3)).astype(np.uint16), rng.randint(0, 256, (n, 3)).astype(np.uint8))
              for n in (600_000, 700_000)]
    for rank in range(world):
        bench.dump_outputs(str(tmp_path), frames, rank=rank, world=world)
    files = list(tmp_path.glob("*.npy"))
    assert len(files) == len(DUMP_NAMES) * world
    total = sum(f.stat().st_size for f in files)
    assert bench.DUMP_POINTS * 40 * 0.99 < total <= 64 << 20


@pytest.mark.gpu
def test_dump_outputs_holds_the_frames_of_the_timed_path(tmp_path):
    """bench.py --dump-outputs on the CUDA path: what it writes for a frame (count, sums, sampled points) equals the oracle's
    frame, for each of the three resident GOFs the kernel-only loop cycles through."""
    import numpy as np
    from oracle import oracle
    from tmc2rs_b200 import abi
    r = run("--steps", "3", "--warmup", "1", "--frames", "8", "--quick", "--no-cpu-baseline", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    files = list(tmp_path.glob("*.npy"))
    assert {f.stem for f in files} == DUMP_NAMES and sum(f.stat().st_size for f in files) <= 64 << 20
    z = {f.stem: np.load(f) for f in files}
    assert all(a.dtype in (np.float32, np.float64) for a in z.values())
    assert len(z["points_per_frame"]) == 3 * 8
    gof, _ = load_bench().build_workload("c2", 8, 8)
    gof.params.geometry_smoothing = gof.params.color_smoothing = True
    view = abi.GofView(gof)
    idx = z["sample_index"].astype(np.int64)
    for f in (0, 5):
        want = oracle.reconstruct_frame(view, f)
        sums = want["positions"].sum(0).tolist() + want["colors"].sum(0).tolist()
        for j in (f, f + 8, f + 16):
            assert z["points_per_frame"][j] == want["point_count"] and z["frame_sums"][j].tolist() == sums
            rows = idx[:, 0] == j
            assert rows.sum() > 1000
            assert np.array_equal(z["sample_positions"][rows], want["positions"][idx[rows, 1]])
            assert np.array_equal(z["sample_colors"][rows], want["colors"][idx[rows, 1]])
