"""Host-side harness logic that needs no GPU: build glue, padding rule, 0/1 check plumbing, summary, CLI."""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from conftest import GOLDEN, REPO
from cuda_l2_b200.harness import correctness as zc
from cuda_l2_b200.harness.common import Padding, kernel_func_name, padding_for, parse_mnk
from tools import utils


@pytest.fixture(scope="module")
def helpers():
    return json.loads((GOLDEN / "helpers.json").read_text())


def test_extract_bm_bk_bn_matches_reference_outputs(helpers):
    for name, text in helpers["snippets"].items():
        assert list(utils.extract_bm_bk_bn(text)) == helpers["extract_bm_bk_bn"][name], name


def test_as_col_major_matches_reference_outputs(helpers):
    for case in helpers["as_col_major"]:
        x = torch.arange(case["rows"] * case["cols"], dtype=torch.float32).reshape(case["rows"], case["cols"]).half()
        y = utils.as_col_major(x)
        assert list(y.shape) == case["shape_out"] and y.is_contiguous() == case["contiguous"]
        assert y.flatten().tolist() == case["flat_out"]
        # storage is the transpose, K-major
        assert torch.equal(y.reshape(case["cols"], case["rows"]), x.t())


def test_build_sources_layout():
    src = utils.get_build_sources("4096_4096_4096", "fp32", "b200")
    assert src == ["cublas/fp32/hgemm_cublas.cu", "cublas/fp32/hgemm_cublaslt_heuristic.cu",
                   "cublas/fp32/hgemm_cublaslt_auto_tuning.cu", "kernels/b200_F32F16F16F32/4096_4096_4096.cu",
                   "pybind/hgemm_b200_fp32.cc"]
    assert utils.get_build_sources("64_64_64", "fp16", "b200")[3] == "kernels/b200_F16F16F16F16/64_64_64.cu"
    for s in src:
        assert (REPO / s).exists(), s
    with pytest.raises(ValueError):
        utils.get_build_sources("64_64_64", "bf16", "b200")
    assert any("compute_100a" in f for f in utils.get_build_cuda_cflags())


def test_kernel_tree_is_complete_and_needs_no_padding():
    grid = (64, 128, 256, 512, 1024, 2048, 4096, 8192, 12288, 16384)
    for d in ("b200_F32F16F16F32", "b200_F16F16F16F16"):
        files = {p.name for p in (REPO / "kernels" / d).glob("*.cu")}
        assert len(files) == 1001
        for m in grid:
            assert f"{m}_{grid[3]}_{grid[-1]}.cu" in files
        assert "2048_11008_4096.cu" in files
    assert padding_for("4096_4096_4096", "fp32", "b200") == Padding(0, 0, 0)
    assert padding_for("64_4096_64", "fp16", "b200") == Padding(0, 0, 0)


def test_padding_rule_with_declared_tiles(tmp_path, monkeypatch):
    # a source that DOES declare tiles gets the reference's padding (benchmarking_offline.py:107-112)
    d = tmp_path / "kernels" / "b200_F32F16F16F32"
    d.mkdir(parents=True)
    (d / "4096_4096_4096.cu").write_text("auto BM = Int<160>{}; \nauto BN = Int<128>{};\nauto BK = Int<32>{};\n")
    import cuda_l2_b200.harness.common as common
    monkeypatch.setattr(common, "PROJECT_DIR", tmp_path)
    assert common.padding_for("4096_4096_4096", "fp32", "b200") == Padding(m=64, k=0, n=0)


def test_parse_and_names():
    assert parse_mnk("2048_11008_4096") == (2048, 11008, 4096)
    for bad in ("1_2", "a_b_c", "0_1_1"):
        with pytest.raises(ValueError):
            parse_mnk(bad)
    assert kernel_func_name("b200", "fp16") == "cuda_l2_b200_fp16"


def test_zero_one_plumbing_passes_and_catches_faults():
    name = "cuda_l2_b200_fp32"
    good = zc.cpu_stand_in(name)
    g = torch.Generator().manual_seed(0)
    res = zc.run_zero_one_check(kernel_funcs=[torch.matmul, good], kernel_under_test_name=name, m=64, n=256, k=64,
                                padding=Padding(), device="cpu", num_iterations=3, generator=g)
    assert res.success and res.result["iterations_run"] == 3 and res.result[f"avg_{name}_diff"] == 0.0

    def off_by_one(a, b, bt, c):
        good(a, b, bt, c)
        c[0, 0] += 1
    off_by_one.__name__ = name
    res = zc.run_zero_one_check(kernel_funcs=[torch.matmul, off_by_one], kernel_under_test_name=name, m=64, n=64, k=64,
                                padding=Padding(), device="cpu", num_iterations=2)
    assert not res.success and "exceeds 0" in res.message

    def scribbler(a, b, bt, c):          # writes one element past the end of C: guard band must notice
        good(a, b, bt, c)
        torch.tensor([], dtype=torch.half).set_(c.untyped_storage(), c.storage_offset() + c.numel(), (1,)).fill_(3.0)
    scribbler.__name__ = name
    res = zc.run_zero_one_check(kernel_funcs=[torch.matmul, scribbler], kernel_under_test_name=name, m=32, n=32, k=32,
                                padding=Padding(), device="cpu", num_iterations=1)
    assert not res.success and "overflow" in res.message

    def nan_maker(a, b, bt, c):
        good(a, b, bt, c)
        c[1, 1] = float("nan")
    nan_maker.__name__ = name
    res = zc.run_zero_one_check(kernel_funcs=[torch.matmul, nan_maker], kernel_under_test_name=name, m=32, n=32, k=32,
                                padding=Padding(), device="cpu", num_iterations=1)
    assert not res.success


def test_zero_one_mask_ignores_large_entries():
    name = "cuda_l2_b200_fp16"

    def saturating(a, b, bt, c):         # wrong only where |truth| > 2047 -> must still pass
        zc.cpu_stand_in(name)(a, b, bt, c)
        c[c > 2047] = 0
    saturating.__name__ = name
    res = zc.run_zero_one_check(kernel_funcs=[saturating], kernel_under_test_name=name, m=4, n=8, k=8192 * 2,
                                padding=Padding(), device="cpu", num_iterations=1)
    assert res.result["levels"] == 3 and res.success


def test_cli_cpu_plumbing_exit_codes(tmp_path):
    cmd = [sys.executable, str(REPO / "zero_one_correctness_check.py"), "--mnk", "64_4096_64", "--acc_precise", "fp32",
           "--device_type", "b200", "--base_dir", str(tmp_path), "--gpu_device_id", "0", "--device", "cpu",
           "--iterations", "2"]
    r = subprocess.run(cmd, cwd=REPO, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    out = json.loads((tmp_path / "zero_one_correctness_check_result.json").read_text())
    assert out["success"] is True and out["result"]["m"] == 64 and out["result"]["n"] == 4096
    bad = subprocess.run(cmd[:-6] + ["--device_type", "a100"], cwd=REPO, capture_output=True, text=True)
    assert bad.returncode != 0      # unknown device type is rejected by argparse


def test_summarize_result_picks_harder_layout(tmp_path):
    import summarize_result as sr
    ours = "cuda_l2_b200_fp32"
    vals = {"hgemm_cublas_tn": (100.0, 120.0), "hgemm_cublas_nn": (90.0, 120.0),
            "hgemm_cublaslt_heuristic_tn": (100.0, 90.0), "hgemm_cublaslt_heuristic_nn": (100.0, 95.0),
            "hgemm_cublaslt_auto_tuning_tn": (110.0, 121.0), "hgemm_cublaslt_auto_tuning_nn": (100.0, 121.0),
            "matmul": (80.0, 120.0)}
    for name, (base, mine) in vals.items():
        (tmp_path / f"benchmark_result_{name}.json").write_text(json.dumps({"records": {name: base, ours: mine}}))
    rows = sr.summarize(str(tmp_path), "fp32", "b200")
    assert rows["cuBLAS-max"]["Baseline TFLOPS"] == 100.0          # tn: speed-up 1.2 < nn 1.33 -> tn is harder
    assert rows["cuBLASLt-heuristic-max"]["Speedup"] == pytest.approx(0.9)
    assert rows["cuBLASLt-auto-tuning-max"]["Speedup"] == pytest.approx(1.1)
    assert rows["torch.matmul"]["Speedup"] == pytest.approx(1.5)
    assert sr.main(["--base_dir", str(tmp_path), "--acc_precise", "fp32", "--device_type", "b200"]) == 0


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` runs on host cores only: one JSON line with the contract's keys."""
    r = subprocess.run([sys.executable, str(REPO / "bench.py"), "--impl", "reference", "--mnk", "256_512_128", "--steps", "2",
                        "--warmup", "1"], cwd=REPO, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["unit"] == "TFLOP/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["config"]["workload"].startswith("256_512_128") and d["steps"] == 2
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_bench_reference_arm_ignores_torchruns_one_thread_default():
    """torchrun exports OMP_NUM_THREADS=1; the reference arm must still use the host's cores (round-1 SCALE ratios at
    N > 1 were inflated ~7.6x by a one-thread reference) and say how many it used."""
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="2", LOCAL_RANK="0")
    r = subprocess.run([sys.executable, str(REPO / "bench.py"), "--impl", "reference", "--mnk", "256_512_128", "--steps", "1",
                        "--warmup", "1", "--gpus", "2"], cwd=REPO, capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    want = max(1, (os.cpu_count() or 2) // 2)
    assert d["cpu_baseline"]["cores"] == want and d["cpu_baseline"]["omp_num_threads_env"] == "1" and d["n_gpus"] == 2
    # a non-zero rank of the reference arm prints nothing and exits 0
    env["RANK"] = "1"
    r = subprocess.run([sys.executable, str(REPO / "bench.py"), "--impl", "reference", "--mnk", "256_512_128", "--steps", "1",
                        "--gpus", "2"], cwd=REPO, capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0 and not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]


def test_bench_sweep_partition_covers_every_shape_once_and_balances():
    import bench
    shapes = bench.sweep_shapes("grid")
    assert len(shapes) == 1001 and (2048, 11008, 4096) in shapes
    for world in (1, 2, 4, 8):
        parts = bench.sweep_partition(shapes, world)
        flat = [s for part in parts for s in part]
        assert sorted(flat) == sorted(shapes) and len(set(flat)) == 1001
        loads = [sum(bench.sweep_cost(s) for s in part) for part in parts]
        assert max(loads) <= 1.02 * (sum(loads) / world) + bench.sweep_cost((16384, 16384, 16384))
    assert bench.sweep_shapes("64_4096_64,4096_4096_4096") == [(64, 4096, 64), (4096, 4096, 4096)]


def test_bench_rejects_a_step_count_below_one_and_a_dump_of_the_cpu_arm(tmp_path):
    base = [sys.executable, str(REPO / "bench.py"), "--impl", "reference", "--mnk", "256_512_128", "--warmup", "1"]
    r = subprocess.run(base + ["--steps", "0"], cwd=REPO, capture_output=True, text=True, timeout=300)
    assert r.returncode == 2 and "at least 1" in r.stderr
    r = subprocess.run(base + ["--steps", "1", "--dump-outputs", str(tmp_path)], cwd=REPO, capture_output=True, text=True,
                       timeout=300)
    assert r.returncode != 0 and "--dump-outputs" in r.stderr and not list(tmp_path.iterdir())


def test_bench_output_sample_is_whole_or_a_fixed_subset():
    import bench
    small = torch.randn(64, 128).half()
    got = bench.output_sample(small)
    assert got.dtype == np.float32 and got.shape == (64, 128) and np.array_equal(got, small.float().numpy())
    big = torch.arange(3000 * 3000, dtype=torch.float32).reshape(3000, 3000)       # each value is its flat index
    got = bench.output_sample(big)
    assert got.dtype == np.float32 and got.ndim == 1 and bench.DUMP_MAX_ELEMS // 2 < got.size <= bench.DUMP_MAX_ELEMS
    assert (np.diff(got) > 0).all() and got[0] >= 0 and got[-1] < big.numel()      # sorted distinct positions
    assert np.array_equal(bench.output_sample(big), got)                            # the same positions every time


def test_bench_without_a_gpu_fails_loudly():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = subprocess.run([sys.executable, str(REPO / "bench.py"), "--steps", "1"], cwd=REPO, capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_attestation_catches_the_five_attacks_of_defense_py():
    """CPU restatement of the reference's self-tests (defense.py:336-579): a legitimate kernel passes, a thread
    spawner, an output replacer / no-op, a dtype changer and a patched timer are each caught."""
    import threading
    import time as _time

    from cuda_l2_b200.harness import attestation as at
    name = "cuda_l2_b200_fp32"
    legit = zc.cpu_stand_in(name)
    a = torch.randn(64, 64).half(); b = torch.randn(64, 64).half()
    bt = utils.as_col_major(b); c = torch.empty(64, 64, dtype=torch.half)
    v = at.attest(legit, a, b, bt, c)
    assert v.passed, v.checks

    stop = threading.Event()
    def spawner(a, b, bt, c):
        legit(a, b, bt, c)
        threading.Thread(target=stop.wait, daemon=True).start()
    v = at.attest(spawner, a, b, bt, c)
    stop.set()
    assert not v.passed and not dict((n, p) for n, p, _ in v.checks)["no_new_threads"]

    v = at.attest(lambda a, b, bt, c: None, a, b, bt, c)                      # never writes c
    assert not dict((n, p) for n, p, _ in v.checks)["real_output"]

    def retyper(a, b, bt, c):
        legit(a, b, bt, c)
        c.data = c.data.float()                                              # "precision downgrade" in reverse: not fp16 any more
    c2 = torch.empty(64, 64, dtype=torch.half)
    v = at.attest(retyper, a, b, bt, c2)
    assert not v.passed

    real = _time.perf_counter
    try:
        _time.perf_counter = lambda: 0.0
        ok, msg = at.check_timers_unpatched()
        assert not ok and "perf_counter" in msg
    finally:
        _time.perf_counter = real
    assert at.check_timers_unpatched()[0]


def test_generated_kernel_sources_compile_for_sm100a(tmp_path):
    """The per-shape translation units the JIT harness builds: one of each flavour (single CTA, CTA pair, multicast
    cluster, cluster split-K, workspace split-K if present, BN = 32) must compile on their own with nvcc."""
    import re
    import shutil
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(nvcc).exists():
        pytest.skip("nvcc not available")
    wanted = {"pair": r"cta_group\*/ 2,", "cluster": r"/\*cluster\*/ (?!1, 1)", "csplit": r"split-K\*/ -", "bn32": r"tile N\*/ 32,",
              "plain": r"cta_group\*/ 1, /\*cluster\*/ 1, 1, /\*group_m\*/ \d+, /\*split-K\*/ 1\)"}
    picked = {}
    for d in ("b200_F32F16F16F32", "b200_F16F16F16F16"):
        for f in sorted((REPO / "kernels" / d).glob("*.cu")):
            text = f.read_text()
            for tag, pat in wanted.items():
                if (d, tag) not in picked and re.search(pat, text):
                    picked[(d, tag)] = f
    assert {t for _, t in picked} == set(wanted), picked.keys()
    for (d, tag), f in list(picked.items())[:8]:
        r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O1", f"-I{REPO}", "-c", str(f),
                            "-o", str(tmp_path / f"{d}_{tag}.o")], capture_output=True, text=True)
        assert r.returncode == 0, (f.name, r.stderr[-1500:])
