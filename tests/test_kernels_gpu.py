"""Numerics of every sm_100a kernel vs a plain PyTorch fp32 reference (run on the B200 box: pytest -m gpu)."""
import pytest
import torch

import paddle_b200 as paddle
from paddle_b200 import kernels
from paddle_b200.kernels import activation as KA
from paddle_b200.kernels import gemm as KG
from paddle_b200.kernels import loss as KL
from paddle_b200.kernels import norm as KN
from paddle_b200.kernels import rope as KR

pytestmark = pytest.mark.gpu


def _ext():
    from paddle_b200._build import ext

    return ext()


def rel_err(a, b):
    a, b = a.float(), b.float()
    return ((a - b).norm() / b.norm().clamp(min=1e-12)).item()


@pytest.mark.parametrize("a_km,b_nk", [(False, False), (False, True), (True, False), (True, True)])
# (512, 300, 256): with b_nk the CTA-pair kernel writes 600-byte output rows, which only its register-store epilogue can handle
@pytest.mark.parametrize("m,n,k", [(256, 512, 256), (384, 320, 192), (128, 64, 64), (1000, 776, 520), (4096, 5120, 1024), (512, 300, 256)])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_gemm_layouts(a_km, b_nk, m, n, k, dtype):
    torch.manual_seed(0)
    dev = "cuda"
    A = torch.randn(m, k, device=dev, dtype=dtype)
    B = torch.randn(k, n, device=dev, dtype=dtype)
    a_in = A.t().contiguous() if a_km else A
    b_in = B.t().contiguous() if b_nk else B
    if not _ext().gemm_supported(a_in, b_in, a_km, b_nk):
        pytest.skip("shape not supported by tcgen05 path")
    out = _ext().gemm(a_in, b_in, None, a_km, b_nk, 0, None, None)
    ref = A.float() @ B.float()
    assert out.shape == (m, n)
    assert rel_err(out, ref) < 5e-3, rel_err(out, ref)


def test_gemm_bias_act_accumulate_fp32out():
    torch.manual_seed(1)
    m, n, k = 512, 768, 384
    A = torch.randn(m, k, device="cuda", dtype=torch.bfloat16)
    B = torch.randn(k, n, device="cuda", dtype=torch.bfloat16)
    bias = torch.randn(n, device="cuda", dtype=torch.bfloat16)
    ref = A.float() @ B.float() + bias.float()
    out = _ext().gemm(A, B, bias, False, False, 1, None, None)
    assert rel_err(out, ref) < 5e-3
    out = _ext().gemm(A, B, bias, False, False, 2, None, None)
    assert rel_err(out, torch.nn.functional.gelu(ref)) < 5e-3
    out = _ext().gemm(A, B, bias, False, False, 3, None, None)
    assert rel_err(out, torch.relu(ref)) < 5e-3
    acc = torch.ones(m, n, device="cuda", dtype=torch.float32)
    _ext().gemm(A, B, None, False, False, 4, acc, None)
    assert rel_err(acc, A.float() @ B.float() + 1) < 1e-3
    o32 = _ext().gemm(A, B, None, False, False, 0, None, torch.float32)
    assert o32.dtype == torch.float32 and rel_err(o32, A.float() @ B.float()) < 1e-3


def test_gemm_batched():
    torch.manual_seed(2)
    b, m, n, k = 6, 256, 192, 128
    A = torch.randn(b, m, k, device="cuda", dtype=torch.bfloat16)
    B = torch.randn(b, n, k, device="cuda", dtype=torch.bfloat16)
    out = _ext().gemm(A, B, None, False, True, 0, None, None)
    ref = torch.einsum("bmk,bnk->bmn", A.float(), B.float())
    assert rel_err(out, ref) < 5e-3


def test_linear_autograd_matches_fp32():
    torch.manual_seed(3)
    x = torch.randn(4, 128, 512, device="cuda", dtype=torch.bfloat16, requires_grad=True)
    w = torch.randn(512, 1024, device="cuda", dtype=torch.bfloat16, requires_grad=True) * 0.05
    w = w.detach().requires_grad_(True)
    b = torch.randn(1024, device="cuda", dtype=torch.bfloat16, requires_grad=True)
    y = KG.linear(x, w, b)
    dy = torch.randn_like(y)
    y.backward(dy)
    xf, wf, bf = x.detach().float().requires_grad_(True), w.detach().float().requires_grad_(True), b.detach().float().requires_grad_(True)
    yr = xf @ wf + bf
    yr.backward(dy.float())
    assert rel_err(y, yr) < 5e-3
    assert rel_err(x.grad, xf.grad) < 5e-3
    assert rel_err(w.grad, wf.grad) < 5e-3
    assert rel_err(b.grad, bf.grad) < 1e-2


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("cols", [512, 5120, 4096, 8192])
def test_rms_norm(dtype, cols):
    torch.manual_seed(0)
    x = torch.randn(300, cols, device="cuda", dtype=dtype, requires_grad=True)
    w = (torch.rand(cols, device="cuda", dtype=dtype) + 0.5).requires_grad_(True)
    y = KN.rms_norm(x, w, 1e-6)
    dy = torch.randn_like(y)
    y.backward(dy)
    xf, wf = x.detach().float().requires_grad_(True), w.detach().float().requires_grad_(True)
    yr = xf * torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + 1e-6) * wf
    yr.backward(dy.float())
    tol = 1e-2 if dtype == torch.bfloat16 else 1e-4
    assert rel_err(y, yr) < tol
    assert rel_err(x.grad, xf.grad) < tol
    assert rel_err(w.grad, wf.grad) < tol * 2


def test_rms_norm_residual():
    x = torch.randn(64, 1024, device="cuda", dtype=torch.bfloat16)
    r = torch.randn_like(x)
    w = torch.rand(1024, device="cuda", dtype=torch.bfloat16)
    y, h = KN.rms_norm(x, w, 1e-6, residual=r)
    hf = (x.float() + r.float())
    assert rel_err(h, hf) < 1e-2
    hh = h.float()
    assert rel_err(y, hh * torch.rsqrt(hh.pow(2).mean(-1, keepdim=True) + 1e-6) * w.float()) < 1e-2


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_layer_norm(dtype):
    torch.manual_seed(0)
    cols = 1024
    x = torch.randn(200, cols, device="cuda", dtype=dtype, requires_grad=True)
    w = (torch.rand(cols, device="cuda", dtype=dtype) + 0.5).requires_grad_(True)
    b = torch.randn(cols, device="cuda", dtype=dtype).requires_grad_(True)
    y = KN.layer_norm(x, [cols], w, b, 1e-5)
    dy = torch.randn_like(y)
    y.backward(dy)
    xf, wf, bf = (t.detach().float().requires_grad_(True) for t in (x, w, b))
    yr = torch.nn.functional.layer_norm(xf, (cols,), wf, bf, 1e-5)
    yr.backward(dy.float())
    tol = 1e-2 if dtype == torch.bfloat16 else 1e-4
    assert rel_err(y, yr) < tol and rel_err(x.grad, xf.grad) < tol
    assert rel_err(w.grad, wf.grad) < 2 * tol and rel_err(b.grad, bf.grad) < 2 * tol


@pytest.mark.parametrize("packed", [False, True])
def test_swiglu(packed):
    g = torch.randn(128, 2048, device="cuda", dtype=torch.bfloat16, requires_grad=True)
    u = torch.randn(128, 2048, device="cuda", dtype=torch.bfloat16, requires_grad=True)
    if packed:
        xin = torch.cat([g.detach(), u.detach()], -1).requires_grad_(True)
        y = KA.swiglu(xin)
    else:
        y = KA.swiglu(g, u)
    dy = torch.randn_like(y)
    y.backward(dy)
    gf, uf = g.detach().float().requires_grad_(True), u.detach().float().requires_grad_(True)
    yr = torch.nn.functional.silu(gf) * uf
    yr.backward(dy.float())
    assert rel_err(y, yr) < 1e-2
    if packed:
        assert rel_err(xin.grad, torch.cat([gf.grad, uf.grad], -1)) < 1e-2
    else:
        assert rel_err(g.grad, gf.grad) < 1e-2 and rel_err(u.grad, uf.grad) < 1e-2


@pytest.mark.parametrize("neox", [True, False])
def test_rope(neox):
    x = torch.randn(2, 64, 8, 128, device="cuda", dtype=torch.bfloat16, requires_grad=True)
    cos, sin = KR.rope_tables(64, 128, device="cuda")
    y = KR.apply_rope(x, cos, sin, None, neox)
    ref = KR.rope_ref(x.detach().float(), cos, sin, None, neox)
    assert rel_err(y, ref) < 1e-2
    dy = torch.randn_like(y)
    y.backward(dy)
    xf = x.detach().float().requires_grad_(True)
    KR.rope_ref(xf, cos, sin, None, neox).backward(dy.float())
    assert rel_err(x.grad, xf.grad) < 1e-2


@pytest.mark.parametrize("vocab", [32000, 1000, 50257])
def test_softmax_ce(vocab):
    torch.manual_seed(0)
    n = 257
    lg = (torch.randn(n, vocab, device="cuda") * 3).to(torch.bfloat16).requires_grad_(True)
    lab = torch.randint(0, vocab, (n,), device="cuda")
    lab[5] = -100
    loss = KL.softmax_cross_entropy(lg, lab, -100)
    w = torch.rand(n, device="cuda")
    (loss * w).sum().backward()
    lf = lg.detach().float().requires_grad_(True)
    lr = torch.nn.functional.cross_entropy(lf, lab, ignore_index=-100, reduction="none")
    (lr * w).sum().backward()
    assert rel_err(loss, lr) < 1e-3
    assert rel_err(lg.grad, lf.grad) < 2e-2


@pytest.mark.parametrize("state_dtype", [torch.float32, torch.bfloat16])
def test_adamw_kernel(state_dtype):
    torch.manual_seed(0)
    n = 100003
    p32 = torch.randn(n, device="cuda")
    g = torch.randn(n, device="cuda").to(torch.bfloat16)
    p = p32.to(torch.bfloat16)
    master = p.float().clone()
    m = torch.zeros(n, device="cuda", dtype=state_dtype)
    v = torch.zeros(n, device="cuda", dtype=state_dtype)
    ref_p = torch.nn.Parameter(master.clone())
    opt = torch.optim.AdamW([ref_p], lr=1e-2, betas=(0.9, 0.95), eps=1e-8, weight_decay=0.1)
    for step in range(1, 4):
        ref_p.grad = g.float()
        opt.step()
        _ext().adamw_step(p, g, master, m, v, 1e-2, 0.9, 0.95, 1e-8, 0.1, step, None, 0.0, None, None)
    tol = 1e-5 if state_dtype == torch.float32 else 2e-2
    assert rel_err(master, ref_p.detach()) < tol
    assert rel_err(p, ref_p.detach()) < 1e-2


def test_grad_norm_and_clip():
    g = torch.randn(1 << 20, device="cuda").to(torch.bfloat16)
    out = torch.zeros(1, device="cuda")
    fi = torch.zeros(1, device="cuda")
    _ext().grad_sq_norm(g, out, fi)
    assert abs(out.item() - g.float().pow(2).sum().item()) / g.float().pow(2).sum().item() < 1e-4
    assert fi.item() == 0
    g[123] = float("inf")
    out.zero_()
    _ext().grad_sq_norm(g, out, fi)
    assert fi.item() == 1


def _attn_ref(q, k, v, causal, scale=None):
    """fp32 reference on [B,S,H,D]."""
    qf, kf, vf = q.float(), k.float(), v.float()
    h, hk = q.shape[2], k.shape[2]
    if hk != h:
        kf, vf = kf.repeat_interleave(h // hk, 2), vf.repeat_interleave(h // hk, 2)
    s = torch.einsum("bqhd,bkhd->bhqk", qf, kf) * (scale or q.shape[-1] ** -0.5)
    if causal:
        sq, sk = q.shape[1], k.shape[1]
        s = s.masked_fill(~torch.ones(sq, sk, dtype=torch.bool, device=q.device).tril(sk - sq), float("-inf"))
    return torch.einsum("bhqk,bkhd->bqhd", s.softmax(-1), vf), torch.logsumexp(s, -1)


@pytest.mark.parametrize("b,s,h,hk,causal", [(2, 512, 4, 4, True), (1, 1024, 2, 2, False), (2, 300, 4, 2, True), (1, 128, 8, 1, False),
                                              (1, 2048, 2, 2, True)])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_flash_attention_fwd(b, s, h, hk, causal, dtype):
    from paddle_b200.kernels import attention as KAT

    torch.manual_seed(0)
    q = torch.randn(b, s, h, 128, device="cuda").to(dtype)
    k = torch.randn(b, s, hk, 128, device="cuda").to(dtype)
    v = torch.randn(b, s, hk, 128, device="cuda").to(dtype)
    assert KAT.fused_ok(q, k, v, None, 0.0, causal)
    n0 = kernels.launch_count()
    out, lse = _ext().attention_fwd(q, k, v, 128 ** -0.5, causal)
    assert kernels.launch_count() == n0 + 1
    ref, ref_lse = _attn_ref(q, k, v, causal)
    assert rel_err(out, ref) < 1e-2, rel_err(out, ref)
    assert (lse - ref_lse).abs().max().item() < 2e-2


def test_flash_attention_packed_views_and_backward():
    """q/k/v as strided views of a packed QKV projection (no split copies); backward vs autograd of the fp32 reference."""
    from paddle_b200.kernels import attention as KAT

    torch.manual_seed(1)
    b, s, nh, nkv = 2, 384, 4, 2
    qkv = (torch.randn(b, s, nh + 2 * nkv, 128, device="cuda") * 0.7).to(torch.bfloat16).requires_grad_(True)
    q, k, v = qkv[:, :, :nh], qkv[:, :, nh:nh + nkv], qkv[:, :, nh + nkv:]
    out = KAT.attention(q, k, v, None, 0.0, True, None)
    g = torch.randn_like(out)
    out.backward(g)
    qkv32 = qkv.detach().float().requires_grad_(True)
    ref, _ = _attn_ref(qkv32[:, :, :nh], qkv32[:, :, nh:nh + nkv], qkv32[:, :, nh + nkv:], True)
    ref.backward(g.float())
    assert rel_err(out, ref) < 1e-2
    assert rel_err(qkv.grad, qkv32.grad) < 2e-2, rel_err(qkv.grad, qkv32.grad)


@pytest.mark.parametrize("b,s,h,hk,causal", [(1, 256, 2, 2, True), (2, 512, 4, 4, True), (1, 384, 4, 2, True), (1, 300, 2, 1, False), (1, 1024, 2, 2, True)])
def test_flash_attention_bwd_kernel(b, s, h, hk, causal):
    """tcgen05 backward kernel vs autograd of the fp32 reference."""
    torch.manual_seed(2)
    q = (torch.randn(b, s, h, 128, device="cuda") * 0.8).to(torch.bfloat16)
    k = (torch.randn(b, s, hk, 128, device="cuda") * 0.8).to(torch.bfloat16)
    v = (torch.randn(b, s, hk, 128, device="cuda") * 0.8).to(torch.bfloat16)
    g = torch.randn(b, s, h, 128, device="cuda").to(torch.bfloat16)
    sc = 128 ** -0.5
    out, lse = _ext().attention_fwd(q, k, v, sc, causal)
    dq, dk, dv = _ext().attention_bwd(q, k, v, out, lse, g, sc, causal)
    q32, k32, v32 = (t.float().requires_grad_(True) for t in (q, k, v))
    ref, _ = _attn_ref(q32, k32, v32, causal)
    ref.backward(g.float())
    assert rel_err(dv, v32.grad) < 2e-2, ("dv", rel_err(dv, v32.grad))
    assert rel_err(dk, k32.grad) < 2e-2, ("dk", rel_err(dk, k32.grad))
    assert rel_err(dq, q32.grad) < 2e-2, ("dq", rel_err(dq, q32.grad))


def test_flash_attention_packed_api():
    """attention_packed: q/k/v read in place from the packed projection, d(qkv) written in place by the backward kernel."""
    from paddle_b200.kernels import attention as KAT

    torch.manual_seed(3)
    b, s, nh, nkv = 1, 640, 4, 4
    qkv = (torch.randn(b, s, nh + 2 * nkv, 128, device="cuda") * 0.7).to(torch.bfloat16).requires_grad_(True)
    out = KAT.attention_packed(qkv, nh, nkv, True, None)
    g = torch.randn_like(out)
    out.backward(g)
    qkv32 = qkv.detach().float().requires_grad_(True)
    ref, _ = _attn_ref(qkv32[:, :, :nh], qkv32[:, :, nh:nh + nkv], qkv32[:, :, nh + nkv:], True)
    ref.backward(g.float())
    assert rel_err(out, ref) < 1e-2
    assert rel_err(qkv.grad, qkv32.grad) < 2e-2, rel_err(qkv.grad, qkv32.grad)


@pytest.mark.parametrize("m,n,k", [(256, 512, 1024), (300, 136, 256), (4096, 5120, 5120)])
@pytest.mark.parametrize("a_dt,b_dt", [(torch.float8_e4m3fn, torch.float8_e4m3fn), (torch.float8_e5m2, torch.float8_e4m3fn)])
def test_gemm_fp8(m, n, k, a_dt, b_dt):
    """tcgen05 kind::f8f6f4 GEMM vs fp32 matmul of the same fp8 values."""
    from paddle_b200.kernels import gemm_fp8 as K8

    torch.manual_seed(0)
    a = (torch.randn(m, k, device="cuda") * 0.5).to(a_dt)
    b = (torch.randn(n, k, device="cuda") * 0.5).to(b_dt)
    bias = torch.randn(n, device="cuda").to(torch.bfloat16)
    out = K8.fp8_gemm(a, b, False, True, bias, 0.37, torch.bfloat16, "relu")
    ref = torch.relu(a.float() @ b.float().t() * 0.37 + bias.float())
    assert rel_err(out, ref) < 1e-2, rel_err(out, ref)
    out2 = K8.fp8_gemm(a, b.t().contiguous(), False, False, None, 1.0, torch.float32)     # non-TN layout -> transposed copy inside
    assert rel_err(out2, a.float() @ b.float().t()) < 1e-3


def test_fp8_linear_training_signal():
    """fp8 Linear (e4m3 fwd, e5m2 grads) tracks the bf16 Linear within fp8 quantisation noise."""
    from paddle_b200.kernels import gemm_fp8 as K8

    torch.manual_seed(1)
    x = (torch.randn(512, 1024, device="cuda")).to(torch.bfloat16).requires_grad_(True)
    w = (torch.randn(1024, 768, device="cuda") * 0.03).to(torch.bfloat16).requires_grad_(True)
    g = torch.randn(512, 768, device="cuda").to(torch.bfloat16)
    y = K8.fp8_linear(x, w)
    y.backward(g)
    x32, w32 = x.detach().float().requires_grad_(True), w.detach().float().requires_grad_(True)
    (x32 @ w32).backward(g.float())
    assert rel_err(y, x32 @ w32) < 6e-2
    assert rel_err(x.grad, x32.grad) < 8e-2 and rel_err(w.grad, w32.grad) < 8e-2


@pytest.mark.parametrize("b,h,hkv,smax", [(2, 8, 8, 777), (3, 16, 4, 2048), (1, 40, 40, 4096)])
def test_decode_attention(b, h, hkv, smax):
    """split-KV decode kernel vs fp32 reference, ragged lengths, GQA."""
    torch.manual_seed(0)
    q = torch.randn(b, h, 128, device="cuda").to(torch.bfloat16)
    kc = torch.randn(b, hkv, smax, 128, device="cuda").to(torch.bfloat16)
    vc = torch.randn(b, hkv, smax, 128, device="cuda").to(torch.bfloat16)
    lens = torch.tensor([smax, max(1, smax // 3), 5][:b], device="cuda", dtype=torch.int32)
    out = _ext().decode_attention(q, kc, vc, lens, 128 ** -0.5)
    rep = h // hkv
    kf, vf = kc.float().repeat_interleave(rep, 1), vc.float().repeat_interleave(rep, 1)
    s = torch.einsum("bhd,bhsd->bhs", q.float(), kf) * 128 ** -0.5
    s = s.masked_fill(torch.arange(smax, device="cuda")[None, None] >= lens[:, None, None], float("-inf"))
    ref = torch.einsum("bhs,bhsd->bhd", s.softmax(-1), vf)
    assert rel_err(out, ref) < 1e-2, rel_err(out, ref)


def test_masked_multihead_attention_uses_decode_kernel():
    import paddle_b200.incubate.nn.functional as IF

    torch.manual_seed(1)
    b, nh, smax = 2, 4, 300
    cache = (torch.randn(2, b, nh, smax, 128, device="cuda") * 0.5).to(torch.bfloat16)
    x = torch.randn(b, 3 * nh * 128, device="cuda").to(torch.bfloat16)
    lens = torch.tensor([17, 250], device="cuda", dtype=torch.int32)
    n0 = kernels.launch_count()
    out, new_cache = IF.masked_multihead_attention(x.as_subclass(paddle.Tensor), cache.clone().as_subclass(paddle.Tensor), sequence_lengths=lens.as_subclass(paddle.Tensor))
    assert kernels.launch_count() > n0
    paddle.set_flags({"FLAGS_use_fused_kernels": True})
    qkv = x.reshape(b, 3, nh, 128).float()
    ck = cache.clone().float()
    bi = torch.arange(b, device="cuda")
    ck[0, bi, :, lens.long()] = qkv[:, 1]
    ck[1, bi, :, lens.long()] = qkv[:, 2]
    s = torch.einsum("bhd,bhsd->bhs", qkv[:, 0], ck[0]) * 128 ** -0.5
    s = s.masked_fill(torch.arange(smax, device="cuda")[None, None] > lens[:, None, None], float("-inf"))
    ref = torch.einsum("bhs,bhsd->bhd", s.softmax(-1), ck[1]).reshape(b, -1)
    assert rel_err(out, ref) < 2e-2


def test_lean_fused_blocks_match_plain_layer():
    """norm->linear / swiglu->linear fused autograd nodes (no saved intermediates) == the plain decoder layer, fwd + all grads."""
    from paddle_b200.models import llama as L

    paddle.set_default_dtype("bfloat16")
    paddle.set_device("gpu:0")
    try:
        paddle.seed(5)
        cfg = L.llama_tiny(hidden_size=256, intermediate_size=512, num_attention_heads=2, num_key_value_heads=2, max_position_embeddings=256)
        layer = L.LlamaDecoderLayer(cfg)
        layer.train()
        h0 = (torch.randn(2, 256, 256, device="cuda") * 2).to(torch.bfloat16)
        g = torch.randn_like(h0)
        res = []
        for lean in (True, False):
            cfg.lean_activations = lean
            for p in layer.parameters():
                p.clear_grad()
            h = h0.clone().as_subclass(paddle.Tensor)
            h.stop_gradient = False
            out = layer(h)
            out.backward(g.as_subclass(paddle.Tensor))
            res.append((out.as_subclass(torch.Tensor).float(), h.grad.as_subclass(torch.Tensor).float(),
                        [p.grad.as_subclass(torch.Tensor).float().clone() for p in layer.parameters()]))
        assert rel_err(res[0][0], res[1][0]) < 1e-2 and rel_err(res[0][1], res[1][1]) < 2e-2
        for a, b in zip(res[0][2], res[1][2]):
            assert rel_err(a, b) < 2e-2
    finally:
        paddle.set_default_dtype("float32")
        paddle.set_device("cpu")


def test_flash_attention_seq_major_layout():
    """Sequence-parallel layout: qkv memory is [S,B,heads,D]; kernels address it through strides, fwd + bwd match the batch-major path."""
    from paddle_b200.kernels import attention as KAT

    torch.manual_seed(4)
    s, b, nh, nkv = 384, 3, 4, 4
    base = (torch.randn(s, b, nh + 2 * nkv, 128, device="cuda") * 0.7).to(torch.bfloat16)
    x_sb = base.clone().requires_grad_(True)
    out_sb = KAT.attention_packed(x_sb, nh, nkv, True, None, seq_major=True)            # [S,B,nh,D]
    g = torch.randn_like(out_sb)
    out_sb.backward(g)
    x_bs = base.transpose(0, 1).contiguous().requires_grad_(True)
    out_bs = KAT.attention_packed(x_bs, nh, nkv, True, None)                            # [B,S,nh,D]
    out_bs.backward(g.transpose(0, 1).contiguous())
    assert rel_err(out_sb.transpose(0, 1), out_bs) < 1e-3
    assert rel_err(x_sb.grad.transpose(0, 1), x_bs.grad) < 1e-2


@pytest.mark.parametrize("lean", [True, False])
def test_fused_wgrad_accumulates_into_arena(lean):
    """Weight gradients of the Llama linears are added straight into the flat gradient arena by the GEMM's accumulate epilogue
    (kernels/wgrad.py); two micro-batches must match the classic autograd accumulation within bf16 rounding."""
    from paddle_b200.kernels import wgrad as WG
    from paddle_b200.models import LlamaForCausalLM, llama_tiny

    paddle.set_device("gpu:0")
    paddle.set_default_dtype("bfloat16")
    try:
        cfg = llama_tiny(hidden_size=512, intermediate_size=1024, num_attention_heads=4, num_key_value_heads=4, num_hidden_layers=2,
                         vocab_size=1024, max_position_embeddings=256, lean_activations=lean)
        ids = paddle.randint(0, cfg.vocab_size, [4, 257])
        grads = {}
        for fused in (True, False):
            paddle.set_flags({"FLAGS_b200_fused_wgrad": fused})
            paddle.seed(5)
            model = LlamaForCausalLM(cfg)
            opt = paddle.optimizer.AdamW(1e-3, parameters=model.parameters(), multi_precision=True)
            opt.enable_flat_arena()
            WG.stats.update(parked=0, fused=0, returned=0)
            for mb in range(2):
                (model(ids[2 * mb:2 * mb + 2, :-1], ids[2 * mb:2 * mb + 2, 1:]) / 2).backward()
            assert (WG.stats["fused"] > 0) == fused, WG.stats
            grads[fused] = {n: p.grad.float().clone() for n, p in model.named_parameters()}
        for n in grads[True]:
            assert rel_err(grads[True][n], grads[False][n]) < 2e-2, (n, rel_err(grads[True][n], grads[False][n]))
    finally:
        paddle.set_flags({"FLAGS_b200_fused_wgrad": True})
        paddle.set_default_dtype("float32")


def test_adamw_split_master_kernel_matches_fp32_master():
    """csrc/optim.cu split master weights (bf16 parameter + int16 residual) == the fp32-master kernel, step after step."""
    from paddle_b200.optimizer.optimizer import split_master_join

    torch.manual_seed(0)
    n = 8 * 4096 + 24
    p0 = (torch.randn(n, device="cuda") * 0.05).to(torch.bfloat16)
    pa, pb = p0.clone(), p0.clone()
    master = p0.float()
    lo = torch.zeros(n, dtype=torch.int16, device="cuda")
    ma, va = torch.zeros(n, device="cuda", dtype=torch.bfloat16), torch.zeros(n, device="cuda", dtype=torch.bfloat16)
    mb, vb = ma.clone(), va.clone()
    e = _ext()
    for step in range(1, 6):
        g = (torch.randn(n, device="cuda") * 0.01).to(torch.bfloat16)
        e.adamw_step(pa, g, master, ma, va, 1e-3, 0.9, 0.95, 1e-8, 0.1, step, None, 0.0, None, None)
        e.adamw_step(pb, g, lo, mb, vb, 1e-3, 0.9, 0.95, 1e-8, 0.1, step, None, 0.0, None, None)
        assert torch.equal(pa, pb), f"parameters diverged at step {step}"
        rebuilt = split_master_join(pb, lo)
        assert (rebuilt.view(torch.int32) - master.view(torch.int32)).abs().max().item() <= 1
    assert lo.abs().max().item() > 0


def test_moe_gate_utility_kernels_match_cpu():
    """number_count / assign_pos / limit_by_capacity / prune_gate_by_capacity on the device (csrc/moe.cu) vs the CPU implementations."""
    from paddle_b200.incubate import moe as M

    torch.manual_seed(0)
    E, n = 8, 5000
    idx = torch.randint(-1, E, (n,))
    c_cpu = M.number_count(idx, E).as_subclass(torch.Tensor)
    c_gpu = M.number_count(idx.cuda(), E).as_subclass(torch.Tensor)
    assert torch.equal(c_cpu, c_gpu.cpu())
    cum = torch.cumsum(c_cpu, 0)
    pos = M.assign_pos(idx.cuda(), cum.cuda()).as_subclass(torch.Tensor).cpu()
    valid = int(c_cpu.sum())
    pos = pos[:valid]
    assert sorted(pos.tolist()) == sorted(torch.nonzero(idx >= 0).reshape(-1).tolist())      # a permutation of the valid tokens ...
    starts = torch.cat([torch.zeros(1, dtype=torch.long), cum[:-1]])
    for e in range(E):                                                                          # ... grouped by expert
        assert bool((idx[pos[starts[e]:cum[e]]] == e).all())
    ec = torch.randint(0, 50, (3 * E,))
    cap = torch.randint(20, 80, (E,))
    assert torch.equal(M.limit_by_capacity(ec, cap, 3).as_subclass(torch.Tensor), M.limit_by_capacity(ec.cuda(), cap.cuda(), 3).as_subclass(torch.Tensor).cpu())
    room = torch.randint(100, 700, (E,))
    g_cpu = M.prune_gate_by_capacity(idx, room, E, 1).as_subclass(torch.Tensor)
    g_gpu = M.prune_gate_by_capacity(idx.cuda(), room.cuda(), E, 1).as_subclass(torch.Tensor).cpu()
    for e in range(E):                                     # same number of survivors per expert (which ones survive is order dependent)
        assert int((g_cpu == e).sum()) == int((g_gpu == e).sum()) == min(int((idx == e).sum()), int(room[e]))
    assert bool(((g_gpu == idx) | (g_gpu == -1)).all())


@pytest.mark.parametrize("act", ["swiglu", "gelu"])
def test_grouped_moe_ffn_matches_per_expert_loop(act):
    """Grouped tcgen05 expert FFN (device routing + 2 grouped GEMM launches) == a per-expert fp32 loop, forward and all gradients."""
    from paddle_b200.kernels import moe as KM

    torch.manual_seed(1)
    T, d, f, E, k = 700, 256, 512, 5, 2
    f1 = 2 * f if act == "swiglu" else f
    x = (torch.randn(T, d, device="cuda") * 0.5).to(torch.bfloat16).requires_grad_(True)
    w1 = (torch.randn(E, d, f1, device="cuda") * 0.05).to(torch.bfloat16).requires_grad_(True)
    w2 = (torch.randn(E, f, d, device="cuda") * 0.05).to(torch.bfloat16).requires_grad_(True)
    logits = torch.randn(T, E, device="cuda")
    val, idx = torch.softmax(logits, -1).topk(k, -1)
    idx = idx.clone()
    idx[::17, 1] = -1                                      # some dropped slots
    idx[:, 0][idx[:, 0] == 3] = 0                          # expert 3 only through the second choice (small), keeps an almost empty expert
    val = val.detach().requires_grad_(True)
    assert KM.grouped_ok(x, w1, w2)
    out = KM.expert_ffn_grouped(x, idx, val, w1, w2, act)
    gout = torch.randn_like(out)
    out.backward(gout)
    got = [t.grad.float().clone() for t in (x, w1, w2, val)]
    xr, w1r, w2r, vr = (t.detach().float().requires_grad_(True) for t in (x, w1, w2, val))
    ref = torch.zeros(T, d, device="cuda")
    for e in range(E):
        for j in range(k):
            sel = torch.nonzero(idx[:, j] == e).reshape(-1)
            if sel.numel() == 0:
                continue
            h = xr[sel] @ w1r[e]
            a = torch.nn.functional.silu(h[:, :f]) * h[:, f:] if act == "swiglu" else torch.nn.functional.gelu(h)
            ref = ref.index_add(0, sel, (a @ w2r[e]) * vr[sel, j:j + 1])
    assert rel_err(out, ref) < 2e-2, rel_err(out, ref)
    ref.backward(gout.float())
    for name, a, b in zip(("dx", "dw1", "dw2", "dval"), got, (xr.grad, w1r.grad, w2r.grad, vr.grad)):
        assert rel_err(a, b) < 3e-2, (name, rel_err(a, b))


@pytest.mark.parametrize("e5m2", [False, True])
def test_fused_fp8_quantize_and_transpose(e5m2):
    """csrc/quant_fp8.cu: amax + cast (+ transposed copy) without a host round trip == the eager per-tensor recipe."""
    torch.manual_seed(2)
    x = (torch.randn(320, 448, device="cuda") * 3).to(torch.bfloat16)
    q, qt, inv = _ext().quantize_fp8(x, e5m2, True)
    fmax = 57344.0 if e5m2 else 448.0
    dt = torch.float8_e5m2 if e5m2 else torch.float8_e4m3fn
    amax = x.float().abs().max()
    ref = (x.float() * (fmax / amax)).clamp(-fmax, fmax).to(dt)
    assert q.dtype == dt and torch.equal(q.float(), ref.float())
    assert torch.equal(qt.float(), ref.float().t())
    assert abs(float(inv) - float(amax / fmax)) < 1e-6 * float(amax / fmax) + 1e-12
    back = q.float() * inv
    assert rel_err(back, x) < (0.15 if e5m2 else 0.05)


def _dense_masked_attention(q, k, v, vis, causal):
    b, sq, h, d = q.shape
    sk = k.shape[1]
    s = torch.einsum("bqhd,bkhd->bhqk", q.float(), k.float()) / d ** 0.5
    m = vis.expand(b, h, sq, sk).clone()
    if causal:
        m &= torch.ones(sq, sk, dtype=torch.bool, device=q.device).tril(sk - sq)
    s = s.masked_fill(~m, float("-inf"))
    p = torch.softmax(s, -1).nan_to_num(0.0)
    return torch.einsum("bhqk,bkhd->bqhd", p, v.float())


@pytest.mark.parametrize("kind", ["flashmask_causal_doc", "flashmask_4", "varlen", "window"])
def test_attention_variants_run_on_own_kernels(kind):
    """flashmask / flash_attn_unpadded / sliding-window attention launch attn::fwd_kernel + the tcgen05 backward (launch counter) and
    match a dense fp32 masked softmax, forward and gradients (reference python/paddle/nn/functional/flash_attention.py:593,1098)."""
    import paddle_b200.nn.functional as F
    from paddle_b200.kernels import attention as KAT

    torch.manual_seed(3)
    B, S, H, D = 2, 384, 4, 128
    mk = lambda *sh: (torch.randn(*sh, device="cuda") * 0.5).to(torch.bfloat16).requires_grad_(True)  # noqa: E731
    causal = False
    if kind == "varlen":
        lens = [100, 180, 104]
        cu = torch.tensor([0, 100, 280, 384], device="cuda", dtype=torch.int32)
        q, k, v = mk(S, H, D), mk(S, H, D), mk(S, H, D)
        causal = True
        kernels.reset_launch_count()
        out, _ = F.flash_attn_unpadded(q.as_subclass(paddle.Tensor), k.as_subclass(paddle.Tensor), v.as_subclass(paddle.Tensor), cu, cu, 180, 180, D ** -0.5, causal=True)
        vis = KAT.colmask_to_dense(KAT.colmask_from_cu_seqlens(cu, cu, S), S)
        ref_in = [t.detach().float().unsqueeze(0) for t in (q, k, v)]
    else:
        q, k, v = mk(B, S, H, D), mk(B, S, H, D), mk(B, S, H, D)
        keys = torch.arange(S, device="cuda")
        if kind == "flashmask_causal_doc":       # causal document mask: two documents per row of the batch
            causal = True
            lts = torch.where(keys < 200, torch.full_like(keys, 200), torch.full_like(keys, S)).reshape(1, 1, S, 1).expand(B, 1, S, 1).int().contiguous()
            se = lts
        elif kind == "flashmask_4":
            lts, lte = (keys + 64).clamp(max=S), (keys + 128).clamp(max=S)
            uts, ute = (keys - 160).clamp(min=0), (keys - 96).clamp(min=0)
            se = torch.stack([lts, lte, uts, ute], -1).reshape(1, 1, S, 4).expand(B, 1, S, 4).int().contiguous()
        kernels.reset_launch_count()
        if kind == "window":
            out = F.flashmask_attention(q.as_subclass(paddle.Tensor), k.as_subclass(paddle.Tensor), v.as_subclass(paddle.Tensor), None, causal=False, window_size=(48, 16))
            vis = KAT.colmask_to_dense(KAT.colmask_from_window(S, S, 48, 16, False, q.device), S)
        else:
            out = F.flashmask_attention(q.as_subclass(paddle.Tensor), k.as_subclass(paddle.Tensor), v.as_subclass(paddle.Tensor), se, causal=causal)
            vis = KAT.colmask_to_dense(KAT.colmask_from_startend(se, causal, S), S)
        ref_in = [t.detach().float() for t in (q, k, v)]
    assert kernels.launch_count() >= 1, "the variant did not reach the native attention kernel"
    out_t = out.as_subclass(torch.Tensor)
    g = torch.randn_like(out_t)
    out_t.backward(g)
    rq, rk, rv = (t.requires_grad_(True) for t in ref_in)
    ref = _dense_masked_attention(rq, rk, rv, vis, causal)
    got = out_t.float().unsqueeze(0) if kind == "varlen" else out_t.float()
    assert rel_err(got, ref) < 2e-2, rel_err(got, ref)
    ref.backward(g.float().unsqueeze(0) if kind == "varlen" else g.float())
    for name, a, b in (("dq", q.grad, rq.grad), ("dk", k.grad, rk.grad), ("dv", v.grad, rv.grad)):
        bb = b.squeeze(0) if kind == "varlen" else b
        assert rel_err(a.float(), bb) < 3e-2, (name, rel_err(a.float(), bb))


@pytest.mark.parametrize("wdt", ["int8", "int4"])
@pytest.mark.parametrize("m", [1, 8, 48, 64])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("k", [1344, 5120])      # 1344 = 21 k-blocks: ragged raw boxes and uneven cluster split-K ranks; 5120: many ring phases
def test_weight_only_linear_dequant_in_sm(wdt, m, dtype, k):
    """csrc/gemm_wo_sm100.cu (raw int8 / int4 weights by TMA, dequantised inside the SM, tcgen05, split-K for decode) vs dequantise + fp32
    matmul; the kernel must be the one that runs (launch counter)."""
    from paddle_b200.nn import quant as Q

    torch.manual_seed(4)
    n = 1536
    w = torch.randn(k, n, device="cuda") * 0.05
    x = (torch.randn(m, k, device="cuda") * 0.5).to(dtype)
    bias = (torch.randn(n, device="cuda") * 0.1).to(dtype)
    wq, sc = Q.weight_quantize(w.as_subclass(paddle.Tensor), algo=f"weight_only_{wdt}")
    kernels.reset_launch_count()
    y = Q.weight_only_linear(x.as_subclass(paddle.Tensor), wq, bias.as_subclass(paddle.Tensor), sc, wdt)
    assert kernels.launch_count() == 1
    wd = Q.weight_dequantize(wq, sc, algo=f"weight_only_{wdt}", out_dtype="float32").as_subclass(torch.Tensor)
    ref = x.float() @ wd.float() + bias.float()
    assert rel_err(y.as_subclass(torch.Tensor), ref) < 1e-2, rel_err(y.as_subclass(torch.Tensor), ref)


def test_mx_quantize_matches_reference():
    """csrc/quant_fp8.cu mx_quantize: e4m3 values and E8M0 block scales equal the PyTorch reference (ceil-rounded power-of-two scale), and
    the 512-byte block layout round-trips through dequantize_mx."""
    from paddle_b200.kernels import gemm_fp8 as G

    torch.manual_seed(2)
    x = (torch.randn(256, 384, device="cuda") * torch.logspace(-3, 2, 384, device="cuda")).to(torch.bfloat16)
    x[5, 32:64] = 0
    q, sf = G.quantize_mx(x)
    # reference on the CPU path of the same function
    qr, sfr = G.quantize_mx(x.cpu())
    assert torch.equal(sf.cpu(), sfr)
    assert torch.equal(q.cpu().view(torch.uint8), qr.view(torch.uint8))
    d = G.dequantize_mx(q, sf)
    dr = G.dequantize_mx(qr, sfr)
    assert torch.equal(d.cpu(), dr)
    assert rel_err(d, x.float()) < 4e-2


@pytest.mark.parametrize("shape", [(128, 128, 128), (256, 384, 512), (384, 1024, 256), (256, 512, 1024)])
@pytest.mark.parametrize("out_dtype", [torch.bfloat16, torch.float32])
def test_mx_block_scaled_gemm(shape, out_dtype):
    """tcgen05.mma.kind::mxf8f6f4.block_scale (csrc/gemm_fp8_sm100.cu, MX): the result equals the fp32 matmul of the DEQUANTISED operands,
    with scales that differ per row and per k-block (a wrong scale slot or byte shows up as an O(1) error)."""
    from paddle_b200.kernels import gemm_fp8 as G

    m, n, k = shape
    torch.manual_seed(7)
    a = torch.randn(m, k, device="cuda") * torch.exp2(torch.randint(-6, 7, (m, k // 32), device="cuda").float()).repeat_interleave(32, 1)
    b = torch.randn(n, k, device="cuda") * torch.exp2(torch.randint(-6, 7, (n, k // 32), device="cuda").float()).repeat_interleave(32, 1)
    aq, sa = G.quantize_mx(a.to(torch.bfloat16))
    bq, sb = G.quantize_mx(b.to(torch.bfloat16))
    bias = torch.randn(n, device="cuda").to(out_dtype)
    kernels.reset_launch_count()
    y = G.mx_gemm(aq, sa, bq, sb, bias, out_dtype)
    assert kernels.launch_count() == 1
    ref = G.dequantize_mx(aq, sa) @ G.dequantize_mx(bq, sb).t() + bias.float()
    tol = 1e-2 if out_dtype == torch.bfloat16 else 1e-5
    assert rel_err(y, ref) < tol, rel_err(y, ref)


def test_mx_fp8_linear_grads():
    """MX block-scaled Linear (three block_scale GEMMs, each quantised along its own contraction axis) vs the fp32 Linear."""
    from paddle_b200.kernels import gemm_fp8 as G

    torch.manual_seed(3)
    x = (torch.randn(256, 512, device="cuda") * 0.5).to(torch.bfloat16).requires_grad_(True)
    w = (torch.randn(512, 384, device="cuda") * 0.05).to(torch.bfloat16).requires_grad_(True)
    b = torch.zeros(384, device="cuda", dtype=torch.bfloat16, requires_grad=True)
    y = G.mx_fp8_linear(x, w, b).as_subclass(torch.Tensor)
    g = torch.randn_like(y)
    y.backward(g)
    xr, wr = x.detach().float().requires_grad_(True), w.detach().float().requires_grad_(True)
    yr = xr @ wr
    yr.backward(g.float())
    assert rel_err(y, yr) < 5e-2
    assert rel_err(x.grad, xr.grad) < 5e-2
    assert rel_err(w.grad, wr.grad) < 5e-2


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_fused_dropout_add_and_bias_dropout_residual_ln(dtype):
    """csrc/fused_dropout.cu: out = dropout(x + bias) + y in one kernel with a byte mask; statistics of the mask, exact reconstruction of the
    forward from it, exact backward, reproducibility under the framework seed, and the fused LayerNorm composition."""
    from paddle_b200.incubate.nn import functional as IF

    x = torch.randn(256, 1024, device="cuda", dtype=dtype, requires_grad=True)
    y = torch.randn(256, 1024, device="cuda", dtype=dtype, requires_grad=True)
    paddle.seed(11)
    kernels.reset_launch_count()
    out = IF.fused_dropout_add(x.as_subclass(paddle.Tensor), y.as_subclass(paddle.Tensor), p=0.25, training=True).as_subclass(torch.Tensor)
    assert kernels.launch_count() == 1
    g = torch.randn_like(out)
    out.backward(g)
    keep = x.grad != 0                                               # the mask, read off the backward (g is never exactly 0)
    kept = keep.float().mean().item()
    assert abs(kept - 0.75) < 0.01, kept
    ref = torch.where(keep, x.detach().float() / 0.75 + y.detach().float(), y.detach().float())
    assert rel_err(out, ref) < (1e-2 if dtype == torch.bfloat16 else 1e-6)
    assert torch.equal(y.grad, g)
    gx_ref = torch.where(keep, g.float() / 0.75, torch.zeros_like(g, dtype=torch.float32))
    assert rel_err(x.grad, gx_ref) < (1e-2 if dtype == torch.bfloat16 else 1e-6)
    paddle.seed(11)
    out2 = IF.fused_dropout_add(x.detach().as_subclass(paddle.Tensor), y.detach().as_subclass(paddle.Tensor), p=0.25, training=True).as_subclass(torch.Tensor)
    assert torch.equal(out2, out.detach())                          # same seed, same masks
    out3 = IF.fused_dropout_add(x.detach().as_subclass(paddle.Tensor), y.detach().as_subclass(paddle.Tensor), p=0.25, training=True).as_subclass(torch.Tensor)
    assert not torch.equal(out3, out2)                              # the generator moved on
    # bias + dropout + residual + LayerNorm
    b = torch.randn(1024, device="cuda", dtype=dtype, requires_grad=True)
    gam = torch.rand(1024, device="cuda", dtype=dtype) + 0.5
    bet = torch.randn(1024, device="cuda", dtype=dtype)
    paddle.seed(5)
    o = IF.fused_bias_dropout_residual_layer_norm(x.detach().as_subclass(paddle.Tensor), y.detach().as_subclass(paddle.Tensor), b.as_subclass(paddle.Tensor),
                                                  gam.as_subclass(paddle.Tensor), bet.as_subclass(paddle.Tensor), dropout_rate=0.1, training=True).as_subclass(torch.Tensor)
    assert abs(o.float().mean().item() - bet.float().mean().item()) < 0.1 and torch.isfinite(o).all()
    o.sum().backward()
    assert b.grad is not None and torch.isfinite(b.grad).all()
    # eval mode is the identity path
    oe = IF.fused_dropout_add(x.detach().as_subclass(paddle.Tensor), y.detach().as_subclass(paddle.Tensor), p=0.25, training=False).as_subclass(torch.Tensor)
    assert rel_err(oe, x.detach().float() + y.detach().float()) < 1e-2


@pytest.mark.parametrize("act", ["gelu", "relu", "silu", "swiglu", "geglu"])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_fused_bias_act_kernel(act, dtype):
    from paddle_b200.incubate.nn import functional as IF

    torch.manual_seed(0)
    x = torch.randn(96, 512, device="cuda", dtype=dtype)
    b = torch.randn(512, device="cuda", dtype=dtype)
    kernels.reset_launch_count()
    out = IF.fused_bias_act(x.as_subclass(paddle.Tensor), b.as_subclass(paddle.Tensor), act_method=act).as_subclass(torch.Tensor)
    assert kernels.launch_count() == 1
    h = x.float() + b.float()
    F = torch.nn.functional
    if act == "swiglu":
        ref = F.silu(h[:, :256]) * h[:, 256:]
    elif act == "geglu":
        ref = F.gelu(h[:, :256]) * h[:, 256:]
    else:
        ref = {"gelu": F.gelu, "relu": torch.relu, "silu": F.silu}[act](h)
    assert out.shape == ref.shape and rel_err(out, ref) < 1e-2


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_paged_block_attention_decode_and_prefill(dtype):
    """incubate/nn/paged_attention.block_attention on CUDA: vectorised cache scatter, decode rows through decode_attention_paged (block-table
    lookups in csrc/decode_attention.cu), prefill rows through the packed varlen tcgen05 attention - against the per-token reference."""
    from paddle_b200.incubate.nn import paged_attention as PA

    torch.manual_seed(0)
    nh, nkv, d, bs, nblocks = 8, 2, 128, 16, 64
    # a mixed batch: two prefill sequences (37 and 130 tokens), three decoding sequences with 5 / 63 / 200 cached positions
    enc = torch.tensor([37, 130, 0, 0, 0], dtype=torch.int32)
    dec = torch.tensor([0, 0, 5, 63, 200], dtype=torch.int32)
    now = torch.tensor([37, 130, 1, 1, 1], dtype=torch.int32)
    cu = torch.zeros(6, dtype=torch.int32)
    cu[1:] = torch.cumsum(now, 0)
    total = int(cu[-1])
    perm = torch.randperm(nblocks)
    bt = torch.full((5, 16), -1, dtype=torch.int32)
    nxt = 0
    for b, need in enumerate([37, 130, 6, 64, 201]):
        n = (need + bs - 1) // bs
        bt[b, :n] = perm[nxt:nxt + n].to(torch.int32)
        nxt += n
    bt = bt.clamp(min=0)
    qkv = (torch.randn(total, (nh + 2 * nkv) * d, device="cuda") * 0.5).to(dtype)
    kc0 = (torch.randn(nblocks, nkv, bs, d, device="cuda") * 0.5).to(dtype)
    vc0 = (torch.randn(nblocks, nkv, bs, d, device="cuda") * 0.5).to(dtype)
    args = (enc.cuda(), dec.cuda(), now.cuda(), cu.cuda(), bt.cuda(), bs)
    kernels.reset_launch_count()
    out, _, kc1, vc1 = PA.block_attention(qkv, kc0.clone(), vc0.clone(), *args)
    assert kernels.launch_count() >= 3                                  # paged decode (2 launches) + varlen attention
    ref, _, kc2, vc2 = PA._block_attention_ref(qkv, kc0.clone(), vc0.clone(), *args)
    assert torch.equal(kc1.as_subclass(torch.Tensor), kc2.as_subclass(torch.Tensor)) and torch.equal(vc1.as_subclass(torch.Tensor), vc2.as_subclass(torch.Tensor))
    o, r = out.as_subclass(torch.Tensor).float(), ref.as_subclass(torch.Tensor).float()
    assert rel_err(o[:167], r[:167]) < 2e-2                             # prefill rows
    assert rel_err(o[167:], r[167:]) < 2e-2                             # decode rows


def test_attention_backward_is_bitwise_reproducible_in_deterministic_mode():
    """FLAGS_cudnn_deterministic: the key tiles reduce into a dQ tile in ascending order (turn counters in csrc/attention_bwd_sm100.cu), so
    repeated backward passes are bit-identical; the default mode (arrival-order bulk reduce) only has to match numerically."""
    E = _ext()
    torch.manual_seed(0)
    b, s, h, d = 2, 1024, 8, 128
    q, k, v = (torch.randn(b, s, h, d, device="cuda", dtype=torch.bfloat16) for _ in range(3))
    out, lse = E.attention_fwd(q, k, v, d ** -0.5, True)
    g = torch.randn_like(out)
    base = E.attention_bwd(q, k, v, out, lse, g, d ** -0.5, True)
    paddle.set_flags({"FLAGS_cudnn_deterministic": True})
    try:
        assert E.deterministic()
        runs = [E.attention_bwd(q, k, v, out, lse, g, d ** -0.5, True) for _ in range(4)]
    finally:
        paddle.set_flags({"FLAGS_cudnn_deterministic": False})
    assert not E.deterministic()
    for r in runs[1:]:
        for a, c in zip(runs[0], r):
            assert torch.equal(a, c)
    for a, c in zip(runs[0], base):
        assert rel_err(a, c.float()) < 2e-2
