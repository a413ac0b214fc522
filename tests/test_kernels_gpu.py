"""Single-kernel parity: each sm_100a kernel, called through the C ABI on device pointers, against a
plain PyTorch fp32 statement of the same op (floating-point kernels keep a torch reference; tolerances
are written next to each check)."""
import ctypes as C
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _check(lib, rc, what):
    assert rc == 0, f"{what}: {lib.b200_last_error().decode()}"


def _cmp(name, got, ref, atol, rtol):
    got, ref = got.float(), ref.float()
    err = (got - ref).abs()
    tol = atol + rtol * ref.abs()
    bad = err > tol
    assert not bad.any(), (f"{name}: {int(bad.sum())}/{bad.numel()} elements out of tolerance; max err "
                           f"{float(err.max()):.5f} at {tuple(int(i) for i in torch.nonzero(err == err.max())[0])}; "
                           f"ref there {float(ref.flatten()[err.argmax()]):.5f} got {float(got.flatten()[err.argmax()]):.5f}; "
                           f"nan={bool(torch.isnan(got).any())}")


def _rand(*shape, scale=1.0, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(torch.bfloat16).to(DEV)


# bf16 output of an fp32-accumulated dot product: error <= 1 bf16 ulp of the result (2^-8 relative) plus
# accumulation-order noise that is far smaller; rtol 2^-7 leaves one ulp of slack.
RTOL = 2.0 ** -7


@pytest.mark.parametrize("M,N,K", [(128, 256, 64), (300, 520, 512), (1000, 1031, 1024), (64, 6144, 4096),
                                   (257, 512, 14336)])
def test_gemm_store(lib, M, N, K):
    A, B = _rand(M, K, seed=1), _rand(N, K, scale=1 / math.sqrt(K), seed=2)
    out = torch.full((M, N), float("nan"), dtype=torch.bfloat16, device=DEV)
    _check(lib, lib.b200_op_gemm(_ptr(A), _ptr(B), _ptr(out), None, M, N, K, 0, 256, 1, N, None), "gemm")
    torch.cuda.synchronize()
    _cmp(f"gemm_store {M}x{N}x{K}", out, A.float() @ B.float().T, 2e-3, RTOL)


def test_gemm_store_residual(lib):
    M, N, K = 200, 512, 1024
    A, B, R = _rand(M, K, seed=1), _rand(N, K, scale=1 / math.sqrt(K), seed=2), _rand(M, N, seed=3)
    out = R.clone()
    _check(lib, lib.b200_op_gemm(_ptr(A), _ptr(B), _ptr(out), _ptr(out), M, N, K, 1, 256, 1, N, None), "gemm")
    torch.cuda.synchronize()
    ref = (A.float() @ B.float().T).to(torch.bfloat16).float() + R.float()
    _cmp("gemm_store_residual", out, ref, 4e-3, RTOL)


def _interleave16(gate, up):
    I, K = gate.shape
    w = torch.empty((2 * I, K), dtype=gate.dtype, device=gate.device)
    w.view(I // 16, 2, 16, K)[:, 0] = gate.view(I // 16, 16, K)
    w.view(I // 16, 2, 16, K)[:, 1] = up.view(I // 16, 16, K)
    return w


def _swiglu_ref(x, gate, up):
    g = (x.float() @ gate.float().T).to(torch.bfloat16)
    u = (x.float() @ up.float().T).to(torch.bfloat16)
    return torch.nn.functional.silu(g.float()).to(torch.bfloat16).float() * u.float()


@pytest.mark.parametrize("M,I,K", [(130, 1024, 512), (64, 2816, 1024)])
def test_gemm_swiglu(lib, M, I, K):
    x = _rand(M, K, seed=1)
    gate, up = _rand(I, K, scale=1 / math.sqrt(K), seed=2), _rand(I, K, scale=1 / math.sqrt(K), seed=3)
    w = _interleave16(gate, up)
    out = torch.full((M, I), float("nan"), dtype=torch.bfloat16, device=DEV)
    _check(lib, lib.b200_op_gemm(_ptr(x), _ptr(w), _ptr(out), None, M, 2 * I, K, 2, 256, 1, I, None), "gemm")
    torch.cuda.synchronize()
    _cmp("gemm_swiglu", out, _swiglu_ref(x, gate, up), 1e-2, 2 * RTOL)


@pytest.mark.parametrize("bn,batch", [(16, 1), (16, 5), (16, 16), (32, 17), (32, 32), (64, 33), (64, 64)])
@pytest.mark.parametrize("nout,K", [(512, 512), (1031, 512), (6144, 4096)])
def test_gemm_swapab_store(lib, bn, batch, nout, K):
    W, x = _rand(nout, K, scale=1 / math.sqrt(K), seed=4), _rand(batch, K, seed=5)
    out = torch.full((batch, nout), float("nan"), dtype=torch.bfloat16, device=DEV)
    _check(lib, lib.b200_op_gemm(_ptr(W), _ptr(x), _ptr(out), None, nout, batch, K, 3, bn, 1, nout, None), "gemm")
    torch.cuda.synchronize()
    _cmp(f"gemm_T_store bn{bn} b{batch}", out, x.float() @ W.float().T, 2e-3, RTOL)


@pytest.mark.parametrize("nout,K,batch,bn", [(28672, 512, 32, 32), (19072, 1024, 5, 16), (128256, 512, 33, 64), (37888, 512, 32, 32),
                                              (4096, 4096, 32, 32), (512, 14336, 32, 32), (6144, 4096, 64, 64), (1031, 512, 7, 16),
                                              (128, 4096, 32, 32), (3584, 4096, 32, 32)])
def test_gemm_streamk_store(lib, nout, K, batch, bn, monkeypatch):
    """Balanced stream-K scheduling with cross-CTA fix-up (two pieces per tile by default; B200_STREAMK_ANY also
    exercises the many-pieces-per-tile path on the small shapes)."""
    monkeypatch.setenv("B200_STREAMK_ANY", "1")
    W, x = _rand(nout, K, scale=1 / math.sqrt(K), seed=4), _rand(batch, K, seed=5)
    for rep in range(3):   # flags must be left clean between launches
        out = torch.full((batch, nout), float("nan"), dtype=torch.bfloat16, device=DEV)
        _check(lib, lib.b200_op_gemm(_ptr(W), _ptr(x), _ptr(out), None, nout, batch, K, 3, bn, 1, nout, None), "gemm")
        torch.cuda.synchronize()
        _cmp(f"gemm_streamk_store rep{rep}", out, x.float() @ W.float().T, 2e-3, RTOL)


@pytest.mark.parametrize("I,K,batch,bn", [(14336, 512, 32, 32), (14336, 1024, 64, 64), (9536, 512, 3, 16)])
def test_gemm_streamk_swiglu(lib, I, K, batch, bn):
    x = _rand(batch, K, seed=1)
    gate, up = _rand(I, K, scale=1 / math.sqrt(K), seed=2), _rand(I, K, scale=1 / math.sqrt(K), seed=3)
    w = _interleave16(gate, up)
    for rep in range(2):
        out = torch.full((batch, I), float("nan"), dtype=torch.bfloat16, device=DEV)
        _check(lib, lib.b200_op_gemm(_ptr(w), _ptr(x), _ptr(out), None, 2 * I, batch, K, 4, bn, 1, I, None), "gemm")
        torch.cuda.synchronize()
        _cmp("gemm_streamk_swiglu", out, _swiglu_ref(x, gate, up), 1e-2, 2 * RTOL)


@pytest.mark.parametrize("bn,batch", [(16, 4), (32, 32), (64, 40)])
def test_gemm_swapab_swiglu(lib, bn, batch):
    I, K = 1024, 512
    x = _rand(batch, K, seed=1)
    gate, up = _rand(I, K, scale=1 / math.sqrt(K), seed=2), _rand(I, K, scale=1 / math.sqrt(K), seed=3)
    w = _interleave16(gate, up)
    out = torch.full((batch, I), float("nan"), dtype=torch.bfloat16, device=DEV)
    _check(lib, lib.b200_op_gemm(_ptr(w), _ptr(x), _ptr(out), None, 2 * I, batch, K, 4, bn, 1, I, None), "gemm")
    torch.cuda.synchronize()
    _cmp("gemm_T_swiglu", out, _swiglu_ref(x, gate, up), 1e-2, 2 * RTOL)


@pytest.mark.parametrize("splits", [1, 2, 3, 4, 7])
@pytest.mark.parametrize("bn,batch", [(16, 3), (32, 32), (64, 64)])
def test_gemm_swapab_splitk(lib, splits, bn, batch):
    nout, K = 512, 1024
    W, x = _rand(nout, K, scale=1 / math.sqrt(K), seed=4), _rand(batch, K, seed=5)
    kb = (K + 63) // 64
    per = -(-kb // splits)
    eff = -(-kb // per)
    ws = torch.full((eff, batch, nout), float("nan"), dtype=torch.float32, device=DEV)
    _check(lib, lib.b200_op_gemm(_ptr(W), _ptr(x), _ptr(ws), None, nout, batch, K, 5, bn, splits, nout, None), "gemm")
    torch.cuda.synchronize()
    _cmp("gemm_T_partial", ws.sum(0), x.float() @ W.float().T, 1e-3, 1e-3)
    # fused consumer: x += bf16(sum partials); xn = rmsnorm(x) * w
    H = nout
    xres, wn = _rand(batch, H, seed=6), (1 + 0.1 * torch.randn(H)).to(torch.bfloat16).to(DEV)
    x2, xn = xres.clone(), torch.empty_like(xres)
    _check(lib, lib.b200_op_rmsnorm(_ptr(x2), _ptr(wn), _ptr(xn), batch, H, 1e-5, _ptr(ws), eff, None, None), "rmsnorm")
    torch.cuda.synchronize()
    xr = (xres.float() + ws.sum(0).to(torch.bfloat16).float()).to(torch.bfloat16)
    assert torch.equal(x2, xr) or (x2.float() - xr.float()).abs().max() <= 2 ** -6 * xr.float().abs().max()
    _cmp("rmsnorm(mode1)", xn, _rmsnorm_ref(x2, wn, 1e-5), 1e-2, RTOL)


def _rmsnorm_ref(x, w, eps):
    xf = x.float()
    var = xf.pow(2).mean(-1, keepdim=True)
    return (w.float() * (xf * torch.rsqrt(var + eps)).to(torch.bfloat16).float())


@pytest.mark.parametrize("rows,H", [(1, 512), (33, 1024), (100, 4096),
                                    (300, 512), (1029, 1024), (4100, 4096), (260, 2048)])   # >= 256 rows: the warp-per-row prefill kernel
def test_rmsnorm(lib, rows, H):
    x, w = _rand(rows, H, scale=3.0, seed=7), (1 + 0.1 * torch.randn(H)).to(torch.bfloat16).to(DEV)
    xn = torch.empty_like(x)
    _check(lib, lib.b200_op_rmsnorm(_ptr(x), _ptr(w), _ptr(xn), rows, H, 1e-5, None, 0, None, None), "rmsnorm")
    torch.cuda.synchronize()
    # same rounding points as LlamaRMSNorm: only the fp32 reduction order differs.  A last-bit difference of the row scale
    # flips bf16(x * rs) by one ulp for ~3e-5 of the elements; with the final rounding of the product that is up to 1.5 ulp
    # on those, so: everything within 2 ulp, and all but 1e-4 of the elements within the 1-ulp bound
    ref = _rmsnorm_ref(x, w, 1e-5)
    _cmp("rmsnorm", xn, ref, 1e-3, 2 * RTOL)
    tight = (xn.float() - ref).abs() <= 1e-3 + RTOL * ref.abs()
    assert float(tight.float().mean()) >= 0.9999
    y = _rand(rows, H, seed=8)
    x2 = x.clone()
    _check(lib, lib.b200_op_rmsnorm(_ptr(x2), _ptr(w), _ptr(xn), rows, H, 1e-5, None, 0, _ptr(y), None), "rmsnorm")
    torch.cuda.synchronize()
    xr = (x.float() + y.float()).to(torch.bfloat16)
    assert torch.equal(x2, xr)
    _cmp("rmsnorm(mode2)", xn, _rmsnorm_ref(xr, w, 1e-5), 1e-3, 2 * RTOL)


def _build_cache(B, lens, nkv, seed):
    """random paged K/V cache with shuffled page ids; returns dense [B][nkv][maxlen][128] views too"""
    max_pages = max((l + 63) // 64 for l in lens) + 1
    num_pages = B * max_pages + 3
    g = torch.Generator().manual_seed(seed)
    perm = torch.randperm(num_pages, generator=g)[: B * max_pages].view(B, max_pages).to(torch.int32)
    kc = torch.zeros((num_pages, nkv, 64, 128), dtype=torch.bfloat16)
    vc = torch.zeros_like(kc)
    maxlen = max(lens)
    kd = torch.zeros((B, nkv, maxlen, 128), dtype=torch.bfloat16)
    vd = torch.zeros_like(kd)
    for b, l in enumerate(lens):
        k = torch.randn((nkv, l, 128), generator=g).to(torch.bfloat16)
        v = torch.randn((nkv, l, 128), generator=g).to(torch.bfloat16)
        kd[b, :, :l], vd[b, :, :l] = k, v
        for p in range((l + 63) // 64):
            n = min(64, l - p * 64)
            kc[perm[b, p], :, :n] = k[:, p * 64:p * 64 + n]
            vc[perm[b, p], :, :n] = v[:, p * 64:p * 64 + n]
    return kc.to(DEV), vc.to(DEV), perm.to(DEV), max_pages, kd.to(DEV), vd.to(DEV)


def _attn_ref(q, k, v, causal_offset=None):
    """q [nh][Lq][128], k/v [nkv][Lk][128] fp32 softmax; returns [Lq][nh*128]"""
    nh, Lq, _ = q.shape
    nkv = k.shape[0]
    G = nh // nkv
    k = k.repeat_interleave(G, 0).float()
    v = v.repeat_interleave(G, 0).float()
    s = (q.float() @ k.transpose(1, 2)) / math.sqrt(128)
    if causal_offset is not None:
        Lk = k.shape[1]
        qi = torch.arange(Lq, device=q.device)[:, None] + causal_offset
        ki = torch.arange(Lk, device=q.device)[None, :]
        s = s.masked_fill(ki > qi, float("-inf"))
    p = torch.softmax(s, -1)
    return (p @ v).transpose(0, 1).reshape(Lq, nh * 128)


@pytest.mark.parametrize("nh,nkv", [(4, 2), (8, 2), (8, 8), (32, 8)])
@pytest.mark.parametrize("lens", [[5], [64, 1, 130], [200, 63, 65, 128, 129], [700, 257]])
def test_attn_prefill_tcgen05(lib, nh, nkv, lens):
    """The tcgen05 / TMEM prefill attention (the engine's) against the fp32 statement of causal GQA attention."""
    B = len(lens)
    kc, vc, pt, max_pages, kd, vd = _build_cache(B, lens, nkv, seed=21)
    T = sum(lens)
    q = _rand(T + 130, nh * 128, seed=22)      # rows beyond T exist so a 128-row TMA box never leaves the buffer
    out = torch.zeros((T, nh * 128), dtype=torch.bfloat16, device=DEV)
    cu = torch.tensor([0] + list(torch.tensor(lens).cumsum(0)), dtype=torch.int32, device=DEV)
    slot = torch.arange(B, dtype=torch.int32, device=DEV)
    _check(lib, lib.b200_op_attn_prefill_tc(_ptr(q), nh * 128, q.shape[0], _ptr(out), nh * 128, _ptr(kc), _ptr(vc), kc.shape[0],
                                            _ptr(pt), max_pages, _ptr(cu), _ptr(slot), B, max(lens), nh, nkv, None), "attn_prefill_tc")
    torch.cuda.synchronize()
    t0 = 0
    for b, l in enumerate(lens):
        qb = q[t0:t0 + l].view(l, nh, 128).transpose(0, 1)
        ref = _attn_ref(qb, kd[b, :, :l], vd[b, :, :l], causal_offset=0)
        _cmp(f"attn_prefill_tc b{b} len{l}", out[t0:t0 + l], ref, 2e-2, 2e-2)
        t0 += l


@pytest.mark.parametrize("nh,nkv", [(4, 2), (8, 2), (32, 8)])
@pytest.mark.parametrize("splits", [1, 2, 5])
def test_attn_decode(lib, nh, nkv, splits):
    lens = [1, 64, 65, 200, 1000, 17]
    B = len(lens)
    kc, vc, pt, max_pages, kd, vd = _build_cache(B, lens, nkv, seed=13)
    q = _rand(B, nh * 128, seed=14)
    slot = torch.arange(B, dtype=torch.int32, device=DEV)
    pos = torch.tensor([l - 1 for l in lens], dtype=torch.int32, device=DEV)
    G = nh // nkv
    po = torch.zeros((B * nkv * splits * G * 128,), dtype=torch.float32, device=DEV)
    pml = torch.zeros((B * nkv * splits * G * 2,), dtype=torch.float32, device=DEV)
    for rep in range(2):   # splits > 1: the last-CTA merge must leave its arrival counters at zero for the next call
        out = torch.zeros((B, nh * 128), dtype=torch.bfloat16, device=DEV)
        _check(lib, lib.b200_op_attn_decode(_ptr(q), nh * 128, _ptr(out), nh * 128, _ptr(kc), _ptr(vc), _ptr(pt), max_pages,
                                            _ptr(slot), _ptr(pos), B, nh, nkv, splits, _ptr(po), _ptr(pml), None), "attn_decode")
        torch.cuda.synchronize()
        for b, l in enumerate(lens):
            qb = q[b].view(nh, 1, 128)
            ref = _attn_ref(qb, kd[b, :, :l], vd[b, :, :l])
            _cmp(f"attn_decode rep{rep} b{b} len{l} splits{splits}", out[b:b + 1], ref, 2e-2, 2e-2)


@pytest.mark.parametrize("T", [70, 4101])      # 4101 tokens: 66 shuffled pages, one CTA per token
def test_rope_kv(lib, T):
    from kserve_b200.engine import hf_rope_tables
    nh, nkv = 4, 2
    npages = (T + 3 + 63) // 64 + 1
    cos, sin = hf_rope_tables(500000.0, 128, npages * 64)
    cosd, sind = cos.to(DEV), sin.to(DEV)
    qkv = _rand(T, (nh + 2 * nkv) * 128, seed=15)
    pos = torch.arange(T, dtype=torch.int32) + 3
    seq = torch.zeros(T, dtype=torch.int32)
    pt = (torch.tensor([[2, 0, 1, 3]], dtype=torch.int32) if T == 70 else
          torch.randperm(npages, generator=torch.Generator().manual_seed(3)).to(torch.int32)[None]).to(DEV)
    kc = torch.zeros((npages if T != 70 else 4, nkv, 64, 128), dtype=torch.bfloat16, device=DEV)
    vc = torch.zeros_like(kc)
    qo = torch.zeros((T, nh * 128), dtype=torch.bfloat16, device=DEV)
    seq_d, pos_d = seq.to(DEV), pos.to(DEV)   # keep alive: the kernel reads them after this call returns
    _check(lib, lib.b200_op_rope_kv(_ptr(qkv), qkv.shape[1], _ptr(qo), nh * 128, _ptr(kc), _ptr(vc), _ptr(pt), pt.shape[1],
                                    _ptr(seq_d), _ptr(pos_d), _ptr(cosd), _ptr(sind), T, nh, nkv, None), "rope")
    torch.cuda.synchronize()
    # HF apply_rotary_pos_emb in bf16 arithmetic (each op rounds), computed with torch on the same device
    c = torch.cat([cosd, cosd], -1)[pos.long().to(DEV)][:, None, :]
    s = torch.cat([sind, sind], -1)[pos.long().to(DEV)][:, None, :]

    def rot(x):
        x1, x2 = x[..., :64], x[..., 64:]
        return torch.cat((-x2, x1), -1)
    qh = qkv[:, : nh * 128].view(T, nh, 128)
    kh = qkv[:, nh * 128:(nh + nkv) * 128].view(T, nkv, 128)
    vh = qkv[:, (nh + nkv) * 128:].view(T, nkv, 128)
    q_ref = (qh * c) + (rot(qh) * s)
    k_ref = (kh * c) + (rot(kh) * s)
    assert torch.equal(qo.view(T, nh, 128), q_ref), "rope(q) not bit-identical to the bf16 HF formula"
    pt_h = pt.cpu()
    for t in (range(T) if T == 70 else list(range(0, T, 37)) + [T - 1, T - 2, T - 3]):
        p = int(pos[t])
        page, slot_ = int(pt_h[0, p // 64]), p % 64
        d = (kc[page, :, slot_].float() - k_ref[t].float()).abs()
        assert torch.equal(kc[page, :, slot_], k_ref[t]), f"k cache mismatch at token {t}: max diff {float(d.max())} n={int((d>0).sum())} page {page} slot {slot_} got {kc[page, 0, slot_, :4].tolist()} ref {k_ref[t][0, :4].tolist()} "
        assert torch.equal(vc[page, :, slot_], vh[t]), f"v cache mismatch at token {t}"


def test_argmax_ties_lowest_index(lib):
    B, V = 5, 128257
    logits = _rand(B, V, seed=16)
    logits[0, 77] = 100.0
    logits[0, 5000] = 100.0   # tie -> lowest index
    logits[1, V - 1] = 50.0
    val = torch.zeros(B, dtype=torch.float32, device=DEV)
    idx = torch.zeros(B, dtype=torch.int32, device=DEV)
    _check(lib, lib.b200_op_argmax(_ptr(logits), V, B, V, _ptr(val), _ptr(idx), None), "argmax")
    torch.cuda.synchronize()
    ref = torch.argmax(logits.float().cpu(), dim=-1)
    assert idx.cpu().tolist() == ref.tolist()
    assert idx[0].item() == 77 and idx[1].item() == V - 1
