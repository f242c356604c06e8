"""CPU-only: the committed bench lines (profiles/r2_bench_n1.json when present, else round 1's; written by `python bench.py` on a
B200) carry every key of the bench contract, and the derived quantities are consistent with each other."""
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _line(name):
  r2 = {"r1_bench_n1_final.json": "r2_bench_n1.json", "r1_bench_reference_arm.json": "r2_bench_reference_arm.json"}.get(name)
  if r2 and os.path.exists(os.path.join(ROOT, "profiles", r2)):
    name = r2
  return json.load(open(os.path.join(ROOT, "profiles", name)))


def test_round2_line_entries():
  """Round-2 additions: every timed region >= 2 s, >= 50 adaptation steps, the other BASELINE.json configurations as keyed entries,
  the CPU baseline measured on the reference's own modules.  A committed r2 line is taken with `bench.py --min-seconds 2`
  (profiles/README.md); with the default (0) every region runs exactly its number of steps."""
  import pytest
  if not os.path.exists(os.path.join(ROOT, "profiles", "r2_bench_n1.json")):
    pytest.skip("no round-2 bench line committed yet")
  d = _line("r1_bench_n1_final.json")
  assert d["steps"] * d["ms_per_step"] >= 1990.0
  assert d["e2e"]["steps"] * d["e2e"]["ms_per_step"] >= 1990.0
  a = d["adapt"]
  assert a["steps"] >= 50 and a["steps"] * a["ms_per_step"] >= 1990.0
  assert abs(a["value"] - 1e3 / a["ms_per_step"]) <= 1e-6 * a["value"]
  sf = d["sceneflow_b32"]
  assert sf["scaling"] == "strong" and abs(sf["value"] - 32e3 / sf["ms_per_batch"]) <= 1e-6 * sf["value"]
  assert len(d["timing_configs"]) >= 5
  assert d["cpu_baseline"]["kind"] == "reference"
  assert "traffic_source" in d["roofline"]


def test_n1_line_has_the_contract_keys():
  d = _line("r1_bench_n1_final.json")
  for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
            "dtype", "data", "config", "e2e", "gpu_launches", "roofline", "cpu_baseline", "clocks"):
    assert k in d, k
  assert d["n_gpus"] == 1 and d["warmup"] >= 3 and d["higher_is_better"] is True and d["scaling"] == "weak"
  assert d["vs_baseline"] is None                      # BASELINE.md holds no published number for this metric
  assert "workload" in d["config"] and "model" not in d["config"]
  assert abs(d["value"] - d["n_gpus"] * 1e3 / d["ms_per_step"]) <= 1e-6 * d["value"]
  e = d["e2e"]
  assert e["h2d_bytes_per_step"] == 2 * 3 * 376 * 1248 * 4 and e["d2h_bytes_per_step"] == 376 * 1248 * 4
  assert 0 < e["value"] <= d["value"] * 1.001          # host copies inside the timed region can only cost time
  assert d["gpu_launches"] == d["launches_per_step"] * d["steps"] > 0
  r = d["roofline"]
  for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
    assert k in r, k
  assert r["bound"] in ("hbm", "tensor") and abs(r["frac"] - r["achieved"] / r["peak"]) <= 1e-9
  c = d["cpu_baseline"]
  assert c["kind"] in ("reference", "port") and c["cores"] >= 1 and c["value"] > 0 and c["sample"]
  assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}


def test_reference_arm_line():
  d = _line("r1_bench_reference_arm.json")
  assert d["impl"] == "reference" and d["metric"] == _line("r1_bench_n1_final.json")["metric"]
  assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
  assert d["cpu_baseline"]["value"] == d["value"]
