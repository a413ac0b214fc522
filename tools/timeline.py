"""Decode-step timeline from the engine's debug trace: per kernel launch (grouped by kind + contiguous time),
start, end, duration, gap to the previous kernel's end."""
import ctypes as C
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench import MODELS, gpu_weights  # noqa: E402
from kserve_b200 import _lib  # noqa: E402
from kserve_b200.engine import B200Engine  # noqa: E402

KIND = {1: "gemm", 2: "rmsnorm", 3: "rope", 4: "attn_dec", 6: "argmax", 7: "step", 8: "embed", 9: "attn_pre", 10: "other"}
EPI = {3: "T_STORE", 4: "T_SWIGLU", 5: "T_PARTIAL", 0: "STORE", 1: "STORE_RES", 2: "SWIGLU"}


def main():
    layers = int(os.environ.get("LAYERS", "4"))
    cfg = dict(MODELS[os.environ.get("MODEL", "llama3_8b")][1], num_hidden_layers=layers)
    B, S, T = 32, 1024, 8
    lib = _lib.load()
    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    nccl_id = None
    if world > 1:
        import torch.distributed as dist
        from kserve_b200.tp import broadcast_nccl_id
        dist.init_process_group("gloo")
        nccl_id = broadcast_nccl_id(rank)
    eng = B200Engine(cfg, max_batch=B, max_seq_len=S + T + 8, max_prefill_tokens=B * S, device=local, tp_rank=rank, tp_size=world,
                     nccl_id=nccl_id)
    eng.load_weights(gpu_weights(cfg, torch.device("cuda", local)))
    ids = torch.randint(3, min(128000, cfg["vocab_size"] - 8), (B, S), dtype=torch.int64)
    eng.stage(ids, None, max_new_tokens=T, pad_token_id=0)
    eng.run_staged(True, 4)          # warm: graph captured
    torch.cuda.synchronize()
    cap = 400000
    _lib.check(lib.b200_debug_trace(cap), "trace")
    if os.environ.get("PHASE", "decode") == "prefill":
        eng.run_staged(True, 0)      # one traced prefill (eager launches, micro-batched under tensor parallelism)
    else:
        eng.run_staged(False, 1)     # one traced decode step (graph replay)
    torch.cuda.synchronize()
    buf = np.zeros((cap, 4), dtype=np.uint64)
    n = C.c_int32()
    _lib.check(lib.b200_debug_trace_read(buf.ctypes.data, cap, C.byref(n)), "read")
    lib.b200_debug_trace(0)
    if rank != 0:
        eng.close()
        return
    rec = buf[: n.value]
    t0, t1 = rec[:, 0].astype(np.int64), rec[:, 1].astype(np.int64)
    tm = rec[:, 2].astype(np.int64)
    kind = (rec[:, 3] & np.uint64(0xFFFFFFFF)).astype(np.int64)
    order = np.argsort(t0)
    t0, t1, kind, tm = t0[order], t1[order], kind[order], tm[order]
    base = t0[0]
    # group consecutive records of the same kind into launches
    launches = []
    for a, b, k, m in zip(t0, t1, kind, tm):
        if launches and launches[-1][0] == k and a <= launches[-1][2] + 20000 and (k % 100) != 0:
            launches[-1][2] = max(launches[-1][2], b)
            launches[-1][3] += 1
            launches[-1][4] = max(launches[-1][4], a)
            if m: launches[-1][5] = min(launches[-1][5], m) if launches[-1][5] else m
            if m: launches[-1][6] = max(launches[-1][6], m)
        else:
            launches.append([k, a, b, 1, a, m, m])
    print(f"{n.value} CTA records, {len(launches)} launches, step span {(t1.max() - base) / 1e3:.1f} us for {layers} layers")
    prev_end = base
    rows = []
    for k, a, b, c, last_start, wmin, wmax in launches:
        name = KIND.get(k % 100, "?")
        if k % 100 == 51:
            name = f"gemm2cta:{EPI.get((k // 100) % 10)}"
        if k % 100 == 1:
            name += f":{EPI.get((k // 100) % 10)}:M{(k // 1000) * 128}"
        rows.append((name, (a - base) / 1e3, (b - base) / 1e3, (b - a) / 1e3, (a - prev_end) / 1e3, c, (last_start - a) / 1e3,
                     (wmin - base) / 1e3 if wmin else -1, (wmax - base) / 1e3 if wmax else -1))
        prev_end = max(prev_end, b)
    per = (len(rows) - 4) // layers if layers else len(rows)
    print("name                          start     end     dur  gap_prev  ctas  cta_start_spread  wait_done(min,max)")
    for r in rows[: int(os.environ.get("ROWS", 2 + 2 * per + 6))]:
        print(f"{r[0]:28s} {r[1]:7.1f} {r[2]:7.1f} {r[3]:7.1f} {r[4]:8.1f} {r[5]:5d} {r[6]:8.1f}   {r[7]:7.1f} {r[8]:7.1f}")
    eng.close()


if __name__ == "__main__":
    main()
