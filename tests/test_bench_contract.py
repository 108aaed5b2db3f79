"""bench.py driver contract: the reference arm always prints one JSON line and exits 0, the
default flags are the BASELINE configuration, the automatic column-slice threshold yields a plan
every rank participates in, and --dump-outputs writes the same arrays from run to run (GPU)."""
import importlib.util
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load_bench():
  spec = importlib.util.spec_from_file_location("de_bench", os.path.join(ROOT, "bench.py"))
  mod = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(mod)
  return mod


def test_reference_arm_prints_one_json_line():
  out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                        "--gpus", "1", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT, check=False)
  assert out.returncode == 0, out.stderr[-2000:]
  lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
  assert len(lines) == 1
  rec = json.loads(lines[0])
  assert rec["impl"] == "reference"
  # either the reference ran (metric/value present) or it says why it could not
  assert "unavailable" in rec or ("metric" in rec and "value" in rec)


def test_defaults_are_the_baseline_config(monkeypatch):
  bench = _load_bench()
  monkeypatch.setattr(sys, "argv", ["bench.py"])
  args = bench.parse_args()
  assert args.gpus == 1 and args.warmup >= 3
  assert args.global_batch == 65536 and args.model == "dlrm-mlperf" and args.dtype == "bf16"
  with open(os.path.join(ROOT, "BASELINE.json"), encoding="utf-8") as f:
    base = json.load(f)
  assert "samples" in json.dumps(base).lower()
  sizes = bench.table_sizes_for("dlrm-mlperf")
  assert len(sizes) == 26 and sum(sizes) == 187767425


@pytest.mark.parametrize("world", [1, 2, 4, 8])
def test_auto_column_slice_threshold(world):
  from distributed_embeddings_b200.parallel.strategy import DistEmbeddingStrategy
  bench = _load_bench()
  sizes = bench.table_sizes_for("dlrm-mlperf")
  thr = bench.auto_column_slice_threshold(sizes, 128, world)
  cfgs = [{"input_dim": s, "output_dim": 128, "combiner": None} for s in sizes]
  st = DistEmbeddingStrategy(cfgs, world, "memory_balanced", column_slice_threshold=thr)
  cols = [sum(st.local_configs[r][m]["output_dim"] for m in st.local_maps[r]) for r in range(world)]
  assert all(c > 0 for c in cols)
  # looked-up columns per rank (what sets gather and NVLink bytes) within 35% of perfect balance
  assert max(cols) <= 1.35 * (26 * 128 / world) + 64
  assert min(c["output_dim"] for r in range(world) for c in st.local_configs[r]) >= 64


def test_step_outputs_sample_the_global_tables():
  """What --dump-outputs writes: the loss, every dense parameter, and the rows of the global
  tables at seeded positions of the batch (here one rank, column-sliced tables)."""
  import numpy as np
  import torch
  from distributed_embeddings_b200.models.dlrm import DLRM
  bench = _load_bench()
  torch.manual_seed(0)
  sizes = [5, 300, 4000, 20]
  model = DLRM(sizes, embedding_dim=16, bottom_mlp_dims=(32, 16), top_mlp_dims=(32, 1),
               device="cpu", compute_dtype=torch.float32, backend="torch",
               column_slice_threshold=1000)
  cat = torch.stack([torch.randint(0, s, (1000,), dtype=torch.int32) for s in sizes])
  out = bench.step_outputs(model, torch.tensor(0.25), cat, 1, 0)
  assert float(out["loss"]) == 0.25
  ids = out["embedding_row_ids"].long().numpy()
  assert ids.shape == (len(sizes), bench.DUMP_ROWS)
  full = model.embedding.get_weights()
  for t in range(len(sizes)):
    np.testing.assert_array_equal(out["embedding_rows"][t].numpy(), full[t][ids[t]])
  dense = {k: p for k, p in model.named_parameters() if not k.startswith("embedding.")}
  assert len(dense) == 8
  for k, p in dense.items():
    assert torch.equal(out[k], p.detach())
  again = bench.step_outputs(model, torch.tensor(0.25), cat, 1, 0)
  assert torch.equal(again["embedding_row_ids"], out["embedding_row_ids"])


@pytest.mark.gpu
def test_dump_outputs_are_reproducible(tmp_path):
  """Two runs with the same flags train on the same inputs: the dumped arrays match."""
  import numpy as np
  n_rows = _load_bench().DUMP_ROWS
  dumps = []
  for run in ("a", "b"):
    out_dir = tmp_path / run
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1",
                          "--steps", "3", "--warmup", "3", "--model", "dlrm-tiny",
                          "--global-batch", "4096", "--no-e2e", "--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT, check=False)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    rec = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert rec["steps"] == 3
    arrays = {p.stem: np.load(p) for p in out_dir.glob("*.npy")}
    assert {"loss", "embedding_rows", "embedding_row_ids", "top_mlp.net.0.weight"} <= set(arrays)
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    assert arrays["embedding_rows"].shape == (26, n_rows, 128)
    assert np.isfinite(arrays["loss"]).all()
    dumps.append(arrays)
  a, b = dumps
  assert a.keys() == b.keys()
  np.testing.assert_array_equal(a["embedding_row_ids"], b["embedding_row_ids"])
  for k in a:
    np.testing.assert_allclose(a[k], b[k], rtol=1e-2, atol=1e-3, err_msg=k)


@pytest.mark.parametrize("world", [2, 4, 8])
def test_default_plan_with_replicated_tables(world):
  """The plan bench.py times by default at N > 1: tables of at most 2500 rows are replicated, the
  column-slice rule only looks at the tables that are still exchanged."""
  from distributed_embeddings_b200.parallel.strategy import DistEmbeddingStrategy
  bench = _load_bench()
  sizes = bench.table_sizes_for("dlrm-mlperf")
  dpt = 2500 * 128
  thr = bench.auto_column_slice_threshold(sizes, 128, world, dpt)
  cfgs = [{"input_dim": s, "output_dim": 128, "combiner": None} for s in sizes]
  st = DistEmbeddingStrategy(cfgs, world, "memory_balanced", column_slice_threshold=thr,
                             data_parallel_threshold=dpt)
  n_dp = len(st.table_groups[0])
  assert n_dp == sum(1 for s in sizes if s * 128 <= dpt) == 11
  assert len(st.table_groups[1]) == 26 - n_dp and not st.table_groups[2]
  cols = [sum(st.local_configs[r][m]["output_dim"] for m in st.local_maps[r]) for r in range(world)]
  assert all(c > 0 for c in cols), "every rank owns part of the exchange"
  mean = (26 - n_dp) * 128 / world
  assert max(cols) <= max(1.25 * mean, mean + 128), (cols, thr)
