"""bench.py host helpers: the algorithmic FLOP model must reproduce SURVEY.md section 8(d)
(29.29 TFLOP per 0.25 degree / 37 level step, 28.81 operational, 4.11 for the 1 degree model),
since `roofline.achieved` and the CPU-sample scaling are defined on it."""
import importlib.util
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bench():
  spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
  mod = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(mod)
  return mod


@pytest.mark.parametrize("workload,tflop", [("graphcast_0.25deg_37lvl", 29.29),
                                            ("graphcast_operational_0.25deg_13lvl", 28.81),
                                            ("graphcast_small_1deg_13lvl", 4.11)])
def test_algorithmic_flops_match_survey(bench, workload, tflop):
  got = bench.algorithmic_flops(*bench.full_workload_sizes(workload)) / 1e12
  assert abs(got - tflop) / tflop < 0.004


def test_thread_candidates(bench):
  assert bench.thread_candidates(128) == [32, 16]        # the oversubscribed 128-thread pass is skipped
  assert bench.thread_candidates(8) == [8]
  assert bench.thread_candidates(48) == [48, 32, 16]


def test_ncu_traffic_reads_the_committed_launch_list():
  import bench
  tc, src = bench.ncu_traffic(bench.DEFAULT_WORKLOAD, "bf16x3")
  assert tc is not None and 100e9 < tc < 250e9           # tensor-core kernels: DRAM bytes per step
  assert "r02_launches_ncu.csv" in src
  assert bench.ncu_traffic("graphcast_small_1deg_13lvl", "bf16x3") == (None, None)


def test_algorithmic_flops_match_the_survey():
  import bench
  f = bench.algorithmic_flops(1038240, 40962, 1618818, 327660, 3114720, 471, 227, 16)
  assert abs(f / 1e12 - 29.29) < 0.01                     # SURVEY.md section 8(d)


def test_dump_outputs_writes_the_whole_output_or_a_fixed_sample(bench, tmp_path, monkeypatch):
  import numpy as np
  import torch
  planes = torch.randn(7, 1000)
  bench.dump_outputs(str(tmp_path / "all"), planes)
  np.testing.assert_array_equal(np.load(tmp_path / "all" / "predictions.npy"), planes.numpy())
  np.testing.assert_array_equal(np.load(tmp_path / "all" / "grid_index.npy"), np.arange(1000))

  monkeypatch.setattr(bench, "DUMP_BYTES", 4096)
  for run in ("a", "b"):
    bench.dump_outputs(str(tmp_path / run), planes)
  files = {run: {n: np.load(tmp_path / run / f"{n}.npy") for n in ("predictions", "grid_index")}
           for run in ("a", "b")}
  idx, pred = files["a"]["grid_index"], files["a"]["predictions"]
  assert idx.dtype == np.float64 and pred.dtype == np.float32
  assert pred.nbytes + idx.nbytes <= 4096 and pred.shape == (7, idx.size) and idx.size > 100
  assert np.all(np.diff(idx) > 0)
  np.testing.assert_array_equal(pred, planes.numpy()[:, idx.astype(np.int64)])
  np.testing.assert_array_equal(files["b"]["grid_index"], idx)
  np.testing.assert_array_equal(files["b"]["predictions"], pred)
