"""The reference-style harness end to end on the B200: JIT-build hgemm_lib for one shape (torch extension with the
reference's 15 exported names), run the 0/1 exactness procedure against every baseline, time one sample."""
import json
import subprocess
import sys

import pytest
import torch

from conftest import REPO

pytestmark = pytest.mark.gpu
EXPORTS = ["init_cublas_handle", "destroy_cublas_handle", "hgemm_cublas_nn", "hgemm_cublas_tn", "init_cublaslt_handle_v1",
           "destroy_cublaslt_handle_v1", "hgemm_cublaslt_heuristic_nn", "hgemm_cublaslt_heuristic_tn",
           "init_cublaslt_handle_v2", "destroy_cublaslt_handle_v2", "find_best_algo_nn_v2_torch",
           "find_best_algo_tn_v2_torch", "hgemm_cublaslt_auto_tuning_nn", "hgemm_cublaslt_auto_tuning_tn"]


@pytest.fixture(scope="module")
def base_dir(tmp_path_factory):
    return tmp_path_factory.mktemp("hgemm_jit")


@pytest.mark.parametrize("acc", ["fp32", "fp16"])
def test_jit_extension_exports_and_passes_zero_one(acc, base_dir):
    from cuda_l2_b200.harness import correctness as zc
    from cuda_l2_b200.harness.common import LibraryHandles, baseline_table, padding_for
    from tools.utils import as_col_major, build_from_sources

    mnk, (m, n, k) = "256_512_1024", (256, 512, 1024)
    hgemm = build_from_sources(mnk=mnk, acc_precise=acc, device_type="b200", base_dir=str(base_dir / acc), verbose=False)
    name = f"cuda_l2_b200_{acc}"
    for sym in EXPORTS + [name]:
        assert hasattr(hgemm, sym), sym
    kernel = getattr(hgemm, name)
    assert kernel.__name__ == name                       # the harness dispatches on this
    pad = padding_for(mnk, acc, "b200")
    assert not pad.any
    with LibraryHandles(hgemm):
        hgemm.find_best_algo_tn_v2_torch(m, n, k)
        hgemm.find_best_algo_nn_v2_torch(m, n, k)
        table = baseline_table(hgemm)
        res = zc.run_zero_one_check(kernel_funcs=[table[x] for x in table] + [kernel], kernel_under_test_name=name,
                                    m=m, n=n, k=k, padding=pad, device="cuda", num_iterations=3)
    assert res.success, res.message
    for key, val in res.result.items():
        if key.startswith("avg_") and key.endswith("_diff"):
            assert val == 0.0, (key, val)                # every library baseline is exact on this domain too
    # error behaviour: C++ exception -> RuntimeError, like the reference's CHECK_TORCH_TENSOR_* macros
    a = torch.zeros((m, k), dtype=torch.half, device="cuda")
    b = torch.zeros((k, n), dtype=torch.half, device="cuda")
    c = torch.zeros((m, n), dtype=torch.half, device="cuda")
    with pytest.raises(RuntimeError):
        kernel(a.float(), b, as_col_major(b), c)
    with pytest.raises(RuntimeError):
        kernel(a, b, as_col_major(b), torch.zeros((m, n + 8), dtype=torch.half, device="cuda"))


def test_offline_benchmark_cli_writes_result(base_dir):
    cmd = [sys.executable, str(REPO / "benchmarking_offline.py"), "--mnk", "256_512_1024", "--acc_precise", "fp32",
           "--device_type", "b200", "--warmup_seconds", "0.2", "--benchmark_seconds", "0.5", "--base_dir",
           str(base_dir / "fp32"), "--gpu_device_id", "0", "--perf_func", "hgemm_cublas_tn"]
    r = subprocess.run(cmd, cwd=REPO, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    rec = json.loads((base_dir / "fp32" / "benchmark_result_hgemm_cublas_tn.json").read_text())["records"]
    assert rec["cuda_l2_b200_fp32"] > 0 and rec["hgemm_cublas_tn"] > 0 and rec["samples"] > 5


def test_server_benchmark_cli_writes_result(base_dir):
    """benchmarking_server.py (reference benchmarking_server.py:144-145: exponential inter-arrival sleeps at --target_qps)
    end to end on one shape, reusing the extension built above."""
    cmd = [sys.executable, str(REPO / "benchmarking_server.py"), "--mnk", "256_512_1024", "--acc_precise", "fp32",
           "--device_type", "b200", "--warmup_seconds", "0.2", "--benchmark_seconds", "0.6", "--base_dir",
           str(base_dir / "fp32"), "--gpu_device_id", "0", "--perf_func", "hgemm_cublaslt_auto_tuning_tn", "--target_qps", "400"]
    r = subprocess.run(cmd, cwd=REPO, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    rec = json.loads((base_dir / "fp32" / "benchmark_result_hgemm_cublaslt_auto_tuning_tn.json").read_text())["records"]
    assert rec["cuda_l2_b200_fp32"] > 0 and rec["hgemm_cublaslt_auto_tuning_tn"] > 0
    # at 400 requests/s for 0.6 s the loop cannot have collected many more than ~240 samples: the sleeps are real
    assert 20 <= rec["samples"] <= 600


def test_bench_runs_the_requested_steps_and_dumps_reproducible_outputs(tmp_path):
    """bench.py times exactly --steps launches, and --dump-outputs writes the same C for the same arguments."""
    import numpy as np
    m, n, k = 256, 512, 1024
    dumps = []
    for run in ("a", "b"):
        cmd = [sys.executable, str(REPO / "bench.py"), "--mnk", f"{m}_{n}_{k}", "--steps", "7", "--warmup", "2",
               "--sweep", "none", "--sustained_seconds", "0", "--e2e_steps", "1", "--cpu_seconds", "0.1",
               "--dump-outputs", str(tmp_path / run)]
        r = subprocess.run(cmd, cwd=REPO, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
        d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        assert d["steps"] == 7 and d["gpu_launches"] == 7
        c = np.load(tmp_path / run / "c.npy")
        assert c.dtype == np.float32 and c.shape == (m, n) and np.isfinite(c).all() and c.std() > 1.0
        dumps.append(c)
    assert np.array_equal(dumps[0], dumps[1])


def test_farm_harness_engine_runs_eval_one_file_for_a_shape(tmp_path):
    """farm_sweep.py --engine harness = the reference-style eval_one_file.sh per shape (0/1 check, one process per
    baseline, summary). Restricted to the cuBLASLt-auto-tuning pair, which is what the sweep's target needs."""
    from cuda_l2_b200 import farm
    rec = farm.run_harness_engine((256, 512, 1024), "fp32", 0.2, 0.6, None, tmp_path, perf_funcs=farm.AUTO_TUNING_PAIR)
    assert rec["ours"] > 0 and rec["lt_auto_tn"] > 0 and rec["lt_auto_nn"] > 0
    assert rec["speedup_vs_lt_auto_max"] == min(rec["lt_auto_tn_speedup"], rec["lt_auto_nn_speedup"])
    assert (tmp_path / "summaries" / "256_512_1024_fp32_offline.json").exists()
    row = farm.speedup_row("256_512_1024", rec)
    assert row["cuBLASLt-auto-tuning-max"] == pytest.approx(rec["speedup_vs_lt_auto_max"]) and row["cuBLAS-max"] == ""


def test_pyharness_engine_times_torch_matmul_and_the_library_pairs(tmp_path):
    """The harness's Python timing loop on the C-ABI libraries (no JIT build): every requested baseline paired with the
    kernel, offline and server pacing, records in the sweep's schema (this is what fills the torch.matmul column)."""
    from cuda_l2_b200 import farm
    out = tmp_path / "worker_fp32_0.jsonl"
    shapes = [(256, 512, 1024), (64, 4096, 64)]
    recs = farm.run_pyharness_worker(0, 1, "fp32", shapes, 0.05, 0.2, None, out,
                                     perf_funcs=("matmul", "hgemm_cublaslt_auto_tuning_tn", "hgemm_cublaslt_auto_tuning_nn"))
    assert len(recs) == 2 and all(r["ok"] for r in recs), recs
    for r in recs:
        assert r["ours"] > 0 and r["matmul"] > 0 and r["lt_auto_tn"] > 0 and r["lt_auto_nn"] > 0
        assert r["speedup_vs_lt_auto_max"] == min(r["lt_auto_tn_speedup"], r["lt_auto_nn_speedup"])
        assert farm.speedup_row(r["mnk"], r)["torch.matmul"] == pytest.approx(r["ours"] / r["matmul"])
    srv = farm.run_pyharness_worker(0, 1, "fp32", shapes[:1], 0.05, 0.3, None, tmp_path / "srv.jsonl",
                                    perf_funcs=("hgemm_cublaslt_auto_tuning_tn",), mode="server", target_qps=200)
    assert srv[0]["ok"] and 5 <= srv[0]["lt_auto_tn_n"] <= 200      # ~60 samples at 200 requests/s for 0.3 s
    assert len(farm.load_done([out])) == 2
