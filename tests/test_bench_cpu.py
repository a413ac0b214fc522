"""bench.py's roofline denominators are the figures of SURVEY.md §8(d), and its helpers behave."""
import json
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402


def test_algorithmic_work_matches_the_survey_figures():
    a = bench.algorithmic(bench.LLAMA3_8B, 32, 1024, 128)
    assert abs(a["layer_params"] - 218_112_000) <= 2 * 4096                # the survey also counts the two norm vectors
    assert abs(a["weight_bytes"] - 15.01e9) < 0.01e9                    # 32 layers + lm_head, bf16
    assert a["kv_bytes_per_token"] == 131_072
    assert abs(a["decode_bytes_per_step"] - 19.57e9) < 0.01e9          # -> 2.98 ms at 6577 GB/s
    assert abs(a["prefill_flops"] - 466e12) < 1e12                      # 457.4 GEMM + 8.8 causal attention + lm_head
    half = bench.algorithmic(bench.LLAMA3_8B, 32, 1024, 128, tp=2)
    assert abs(half["decode_bytes_per_step"] * 2 - a["decode_bytes_per_step"]) < 1 and abs(half["prefill_flops"] * 2 - a["prefill_flops"]) < 1
    m = bench.algorithmic(bench.MIXTRAL_8X7B, 32, 1024, 128, tp=4)
    assert abs(m["weight_bytes"] * 4 - 93.4e9) < 0.5e9                  # all 8 experts stream (46.7 B params incl. the embedding)


def test_traffic_comes_from_the_committed_capture_only_on_its_configuration():
    t = bench.ncu_decode_traffic(bench.LLAMA3_8B, 32, 1024, 128, 1)
    a = bench.algorithmic(bench.LLAMA3_8B, 32, 1024, 128)["decode_bytes_per_step"]
    assert t is not None and 1.0 <= t / a < 1.1                         # no wasted re-reads
    assert bench.ncu_decode_traffic(bench.LLAMA3_8B, 64, 1024, 128, 1) is None
    assert bench.ncu_decode_traffic(bench.LLAMA3_8B, 32, 1024, 128, 2) is None
    assert bench.ncu_decode_traffic(bench.MIXTRAL_8X7B, 32, 1024, 128, 1) is None


def test_cpu_thread_policy_and_peaks():
    n = bench.usable_cores()
    assert 1 <= n <= (os.cpu_count() or 1)
    p = bench.load_peaks()
    assert p["hbm_gbs"] > 1000 and p["tf_sustained"] <= p["tf_burst"]
    assert json.dumps(p)


def test_dump_outputs_writes_exact_float64_ids(tmp_path, monkeypatch):
    ids = torch.randint(0, 128256, (4, 9), generator=torch.Generator().manual_seed(0), dtype=torch.int64)
    bench.dump_outputs(str(tmp_path / "out"), {"output_ids": ids})
    a = np.load(tmp_path / "out" / "output_ids.npy")
    assert a.dtype == np.float64 and a.shape == (4, 9) and np.array_equal(a.astype(np.int64), ids.numpy())
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", ids.numel() * 8 - 1)
    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path / "big"), {"output_ids": ids})
    assert not (tmp_path / "big").exists()


def test_both_arms_share_one_config_dict():
    """VERDICT r01: the reference arm mislabelled its workload and `same_config` was false.  Both arms now build `config`
    from one function of (model, batch, prompt, gen, gpus), and it states what one reference step is."""
    a = bench.workload_config("Llama-3-8B", 32, 1024, 128, 4)
    assert a == bench.workload_config("Llama-3-8B", 32, 1024, 128, 4)
    assert a["global_batch"] == 32 and a["parallelism"] == "tp4" and "batch 1 x 1024-in/128-out in full" in a["reference_sample"]
    src = open(bench.__file__).read()
    assert src.count('"config": workload_config(') == 2          # the GPU arm and the reference arm, nothing hand-written
