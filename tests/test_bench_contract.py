"""bench.py contract checks that need no GPU: the reference arm (CPU port) prints the agreed JSON line, and the
product arm refuses to run without a CUDA device (there is no CPU fallback to time by accident)."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]


def _run(*args, env=None):
    return subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, cwd=ROOT,
                          timeout=600, env=env)


def test_reference_arm_json_line():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0", "--catalog-rows", "20000", "--nq", "16", "--topk", "10")
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["unit"] == "queries/s" and line["higher_is_better"] is True
    assert line["n_gpus"] == 1 and line["steps"] == 1 and line["warmup"] == 0 and line["value"] > 0
    assert line["config"]["workload"] == "flat_ip_top10_20000x384_nq16"
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["cpu_baseline"]["value"] == line["value"]
    assert line["metric"] == "exact top-10 queries/s, 20000x384 catalog"
    assert line["extrapolated"]["is_extrapolated"] is False and line["extrapolated"]["sample_rows"] == 20000
    assert line["e2e"] == {"value": line["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["vs_baseline"] is None and line["gpu_launches"] == 0


def test_product_arm_needs_cuda():
    if torch.cuda.is_available():
        return
    r = _run("--steps", "1", "--catalog-rows", "20000", "--nq", "16")
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_bad_steps_and_dump_of_the_cpu_arm_are_refused():
    r = _run("--impl", "reference", "--steps", "0", "--warmup", "0", "--catalog-rows", "20000", "--nq", "16")
    assert r.returncode != 0 and "--steps" in r.stderr
    r = _run("--impl", "reference", "--steps", "1", "--catalog-rows", "20000", "--nq", "16", "--dump-outputs", "x")
    assert r.returncode != 0 and "--dump-outputs" in r.stderr


def test_dump_outputs_dtypes_and_bounded_sample(tmp_path, monkeypatch):
    """scores stay float32, ids become float64 (exact below 2**53); a result above the size cap is cut to a fixed
    seeded sample of query rows, listed in rows.npy."""
    sys.path.insert(0, str(ROOT))
    import bench
    s = torch.rand(50, 7)
    i = torch.randint(0, 1 << 40, (50, 7))
    bench.dump_outputs(tmp_path / "full", s, i)
    assert sorted(p.name for p in (tmp_path / "full").iterdir()) == ["ids.npy", "scores.npy"]
    gs, gi = np.load(tmp_path / "full" / "scores.npy"), np.load(tmp_path / "full" / "ids.npy")
    assert gs.dtype == np.float32 and gi.dtype == np.float64
    assert np.array_equal(gs, s.numpy()) and np.array_equal(gi.astype(np.int64), i.numpy())
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 4096 + 10 * (7 * 12 + 8))
    for name in ("a", "b"):
        bench.dump_outputs(tmp_path / name, s, i)
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert rows.dtype == np.float64 and len(rows) == 10 and np.all(np.diff(rows) > 0)
    assert np.array_equal(rows, np.load(tmp_path / "b" / "rows.npy"))
    r = rows.astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "a" / "scores.npy"), s.numpy()[r])
    assert np.array_equal(np.load(tmp_path / "a" / "ids.npy").astype(np.int64), i.numpy()[r])


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_batch_and_repeats(tmp_path):
    """--dump-outputs writes the results of the last timed step (checked against the fp32 torch checker on the same
    seeded catalog and queries), and a second run with the same arguments writes the same bytes."""
    args = ["--steps", "2", "--warmup", "3", "--catalog-rows", "20000", "--nq", "16", "--topk", "10", "--no-secondary"]
    for name in ("a", "b"):
        r = _run(*args, "--dump-outputs", str(tmp_path / name))
        assert r.returncode == 0, r.stderr[-2000:]
    for f in ("scores.npy", "ids.npy"):
        assert (tmp_path / "a" / f).read_bytes() == (tmp_path / "b" / f).read_bytes(), f
    s, i = np.load(tmp_path / "a" / "scores.npy"), np.load(tmp_path / "a" / "ids.npy")
    assert s.dtype == np.float32 and i.dtype == np.float64 and s.shape == i.shape == (16, 10)
    sys.path.insert(0, str(ROOT))
    import bench
    index, _, _ = bench.make_shard(20000, 384, 1, 0)
    q = torch.randn((5, 16, 384), device="cuda", generator=torch.Generator(device="cuda").manual_seed(4321))[4]
    ts, ti = bench.torch_flat_topk(index.xn, q, 10)
    rep = bench.compare_topk_device(torch.from_numpy(s).cuda(), torch.from_numpy(i).long().cuda(), ts, ti)
    assert rep["ok"], rep


def test_reference_arm_under_torchrun_uses_all_threads_and_is_bounded():
    """The driver launches the reference arm like the product arm (torchrun for N > 1), and torchrun exports
    OMP_NUM_THREADS=1: rank 0 must still use every host core, sample the catalog to its time budget, say that the
    number is extrapolated, and the other ranks must exit 0 without printing a line."""
    import os
    import socket
    import time
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    env = dict(os.environ, TT_BENCH_REF_BUDGET_S="4")
    env.pop("OMP_NUM_THREADS", None)
    t = time.time()
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), str(ROOT / "bench.py"),
                        "--impl", "reference", "--gpus", "2", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, cwd=ROOT, timeout=300, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [json.loads(l) for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, "only rank 0 prints"
    line = lines[0]
    ncpu = len(os.sched_getaffinity(0))
    assert line["cpu_baseline"]["cores"] == ncpu, "torchrun's OMP_NUM_THREADS=1 must not throttle the CPU arm"
    assert line["n_gpus"] == 2 and line["config"]["workload"] == "flat_ip_top100_10000000x384_nq4096"
    assert line["metric"] == "exact top-100 queries/s, 10Mx384 catalog"
    ex = line["extrapolated"]
    assert ex["is_extrapolated"] and "extrapolated" in line["dtype"] and "EXTRAPOLATED" in line["cpu_baseline"]["sample"]
    assert abs(line["ms_per_step"] - ex["measured_ms_per_sample_step"] * ex["scale"]) < 1e-6 * line["ms_per_step"]
    assert time.time() - t < 120


def test_parity_comparator_tie_rules():
    """bench.compare_topk_device: score errors, swaps inside / outside ties and boundary ties."""
    sys.path.insert(0, str(ROOT))
    import bench
    rs = torch.tensor([[0.9, 0.8, 0.7, 0.6]])
    ri = torch.tensor([[10, 11, 12, 13]])
    assert bench.compare_topk_device(rs.clone(), ri.clone(), rs, ri)["ok"]
    assert not bench.compare_topk_device(rs + 2e-5, ri, rs, ri)["ok"]                       # score tolerance
    sw = torch.tensor([[10, 12, 11, 13]])
    assert not bench.compare_topk_device(rs, sw, rs, ri)["ok"]                              # swap across a 0.1 gap
    rt = torch.tensor([[0.9, 0.8, 0.8 - 5e-7, 0.6]])
    assert bench.compare_topk_device(rt, sw, rt, ri)["ok"]                                  # swap inside a tie
    other = torch.tensor([[10, 11, 12, 99]])
    assert bench.compare_topk_device(rs, other, rs, ri)["ok"]                               # boundary tie (same score)
    assert not bench.compare_topk_device(rs - torch.tensor([[0, 0, 0, 5e-6]]), other, rs, ri)["ok"]


def test_clock_sampler_keeps_only_samples_of_the_timed_region():
    """bench.ClockSampler.summary: samples stamped outside [enter, exit] are dropped (nvidia-smi starts before the timed
    region and runs past it); a region shorter than one sampling period falls back to the first samples after its start."""
    sys.path.insert(0, str(ROOT))
    import bench
    row = "{sm}, 1965, 700.0, Not Active, Not Active, Not Active, {cap}\n"
    cs = bench.ClockSampler(0)
    cs.t0, cs.t1 = 10.0, 11.0
    cs.lines = [(9.5, row.format(sm=300, cap="Not Active")), (10.2, row.format(sm=1650, cap="Active")),
                (10.6, row.format(sm=1700, cap="Active")), (11.5, row.format(sm=200, cap="Not Active"))]
    out = cs.summary()
    assert out["samples"] == 2 and out["sm_mhz"] == 1675.0 and out["sm_max_mhz"] == 1965.0
    assert out["reasons"] == ["sw_power_cap"]
    cs.t0, cs.t1 = 10.0, 10.01                       # 10 ms region: no sample inside
    cs.lines = [(9.9, row.format(sm=300, cap="Not Active")), (10.05, row.format(sm=1900, cap="Not Active"))]
    out = cs.summary()
    assert out["samples"] == 1 and out["sm_mhz"] == 1900.0 and out["reasons"] == []
    cs.lines = []
    assert cs.summary()["sm_mhz"] is None
