"""bench.py's CPU legs (the reference's own kernels timed beside the GPU numbers) run on any host: shapes of what they return, bounded run time.
The GPU arm itself needs a B200 (tests/test_gpu_*.py); the reference arm under torchrun is covered by tests/test_dist_gloo.py."""
import importlib.util
import json
import time
from pathlib import Path

import pytest

from oracle import capi

ROOT = Path(__file__).resolve().parents[1]
needs_reference_avx = pytest.mark.skipif(not capi.ref_available("avx"), reason="reference AVX build (oracle/_ref) not present")


@pytest.fixture(scope="module")
def bench():
    spec = importlib.util.spec_from_file_location("bench_module", ROOT / "bench.py")
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


@needs_reference_avx
def test_w8a8_cpu_baseline_leg(bench):
    t0 = time.perf_counter()
    d = bench.cpu_baseline_w8a8(0.5)
    assert time.perf_counter() - t0 < 120
    json.dumps(d)  # plain Python numbers only: it is embedded in the bench line
    assert d["kind"] == "reference" and d["cores"] >= 1 and d["ms_per_layer_linears"] > 0
    # 157 MB of int8 weights per layer
    assert abs(d["weight_GB_per_s"] * d["ms_per_layer_linears"] * 1e6 - (4 * 4096 * 4096 + 2 * 4096 * 11008)) < 1e3


@needs_reference_avx
def test_prefill_cpu_baseline_leg(bench):
    d = bench.cpu_baseline_prefill(2, model="tiny-gqa", m=32)
    json.dumps(d)
    assert d["kind"] == "reference" and d["rows"] == 32 and d["s_per_layer_linears"] > 0 and "estimate" in d["sample"]
    assert d["tok_per_s_scaled"] == pytest.approx(32 / (d["s_per_layer_linears"] * 2))  # tiny-gqa has 2 layers


def test_both_arms_name_the_same_workload(bench):
    """The `config` object is built by one function for both arms: identical keys and values (the driver compares them)."""
    import argparse

    from tinychatengine_b200.llama import GEOMETRIES

    a = argparse.Namespace(max_ctx=4096, ctx=-1)
    g = GEOMETRIES["llama3-8b"]
    c1, c2 = bench.workload_config(g, a, 1, False), bench.workload_config(g, a, 1, False)
    assert c1 == c2 and set(c1) == {"workload", "sequences", "max_ctx", "parallelism"} and "model" not in c1
    assert bench.workload_config(g, a, 8, True)["parallelism"] != c1["parallelism"]
