"""Every CUDA kernel behind the C ABI against a plain torch fp32 reference of the same op (autograd for
the backward kernels), plus the integer token path against the numpy oracle (bit-exact)."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda"


def rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


@pytest.fixture(scope="module")
def lib():
    from open_musiclm_b200 import lib as L
    L.device_check()
    return L


# ------------------------------------------------------------------------------------------------ integer path
@pytest.mark.parametrize("with_pad", [False, True])
def test_token_plan_bit_exact(lib, with_pad):
    from oracle import restatement as R
    cfg = R.coarse_cfg(codebook=1024, n_clap_q=12, n_coarse_q=3)
    g = torch.Generator().manual_seed(5)
    toks = [torch.randint(0, 1024, s, generator=g) for s in [(3, 12), (3, 40), (3, 17, 3)]]
    if with_pad:  # pads (-1) in every sequence: only recognised at quantizer-0 positions after the offset add
        toks[0][0, 0] = -1; toks[0][1, 5] = -1; toks[1][2, 3] = -1; toks[2][0, 0, 0] = -1; toks[2][1, 2, 1] = -1
    ids_np, mask_np, labels_np = R.prepare_ids(cfg, [t.numpy() for t in toks], True)
    rows = R.embedding_rows(cfg, ids_np)
    bases = [0, 1025 * 12, 1025 * 12 + 1025]
    total_rows = bases[2] + 1025 * 3
    ids_out, src_row, key_mask, labels, n_tok = lib.token_plan(
        [t.to(DEV) for t in toks], [1024] * 3, [12, 1, 3], bases, [total_rows, total_rows + 1, total_rows + 2],
        append_eos=True, drop_last=True, mask_cond=True)
    assert np.array_equal(ids_out.cpu().numpy(), np.concatenate(ids_np, 1))
    assert np.array_equal(key_mask.cpu().numpy().astype(bool), mask_np)
    assert np.array_equal(labels.cpu().numpy(), np.concatenate(labels_np, 1).astype(np.int32))
    exp = []
    for s, (r, pad) in enumerate(rows):
        exp.append(np.full((3, 1), total_rows + s))
        exp.append(np.where(pad, -1, r + bases[s]))
    assert np.array_equal(src_row.cpu().numpy(), np.concatenate(exp, 1).astype(np.int32))


def test_forgetful_mask_properties(lib):
    B, N = 16, 1024
    seed = torch.tensor([12345], dtype=torch.int64, device=DEV)
    k = min(int(N * 0.15), N - 1)
    keep = lib.forgetful_mask(B, N, k, seed, 7, DEV).cpu().numpy()
    assert keep[:, 0].all()
    assert ((keep == 0).sum(1) == k).all()
    keep2 = lib.forgetful_mask(B, N, k, seed, 8, DEV).cpu().numpy()
    assert (keep != keep2).any()
    assert not np.array_equal(keep[0], keep[1])
    # roughly uniform over positions 1..N-1
    many = np.stack([lib.forgetful_mask(B, N, k, seed, 100 + i, DEV).cpu().numpy() for i in range(20)])
    freq = 1.0 - many[:, :, 1:].mean((0, 1))
    assert abs(freq.mean() - k / (N - 1)) < 1e-6 and freq.max() < 0.3 and freq.min() > 0.05


def test_embed_gather_scatter(lib):
    torch.manual_seed(0)
    table = torch.randn(500, 256, device=DEV)
    src = torch.randint(-1, 500, (64,), device=DEV, dtype=torch.int32)
    x = torch.empty(64, 256, device=DEV)
    lib.embed_gather(table, src, x)
    ref = torch.where((src >= 0)[:, None], table[src.clamp_min(0).long()], torch.zeros(1, device=DEV))
    assert torch.equal(x, ref)
    src2 = torch.randint(-1, 500, (64,), device=DEV, dtype=torch.int32)      # second row (absolute position embeddings)
    lib.embed_gather(table, src, x, src2)
    ref2 = ref + torch.where((src2 >= 0)[:, None], table[src2.clamp_min(0).long()], torch.zeros(1, device=DEV))
    assert torch.equal(x, ref2)
    dx = torch.randn(64, 256, device=DEV)
    dt = torch.zeros_like(table)
    lib.embed_scatter_add(dt, src, dx, 0.1)
    ref_dt = torch.zeros_like(table).index_add_(0, src.clamp_min(0).long(), dx * 0.1 * (src >= 0)[:, None])
    assert rel(dt, ref_dt) < 1e-6


# ------------------------------------------------------------------------------------------------ norms
@pytest.mark.parametrize("ydt", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("M,D", [(100, 64), (77, 128), (513, 1024), (33, 192)])
def test_layernorm_fwd_bwd(lib, M, D, ydt):
    torch.manual_seed(M + D)
    x = (torch.randn(M, D, device=DEV) * 3 + 0.5).requires_grad_(True)
    gamma = (1 + 0.2 * torch.randn(D, device=DEV)).requires_grad_(True)
    y = torch.empty(M, D, device=DEV, dtype=ydt)
    xr = torch.empty(M, D, device=DEV, dtype=torch.bfloat16)
    stats = torch.empty(M, 2, device=DEV)
    yc = torch.empty(M, D, device=DEV, dtype=torch.bfloat16)
    lib.layernorm_fwd(x.detach(), gamma.detach(), y, xr, stats, ycopy=yc)
    ref = F.layer_norm(x, (D,), gamma, None, 1e-5)
    assert rel(yc, ref.detach()) < 4e-3 and (ydt != torch.bfloat16 or torch.equal(yc, y))
    assert rel(y, ref.detach()) < (4e-3 if ydt == torch.bfloat16 else 5e-4)
    assert torch.equal(y, ref.detach().to(ydt)) or rel(y, ref.detach().to(ydt)) < 1e-3     # same rounding as torch's cast (up to fp32 ulps)
    assert torch.equal(xr, x.detach().bfloat16())
    dy = torch.randn(M, D, device=DEV).bfloat16()
    dres = torch.randn(M, D, device=DEV)
    draw = torch.randn(M, D, device=DEV).bfloat16()
    ref.backward(dy.float())
    dx = torch.empty(M, D, device=DEV)
    dgamma = torch.zeros(D, device=DEV)
    lib.layernorm_bwd(dy, x.detach(), stats, gamma.detach(), dx, dgamma, dres=dres, draw=draw)
    assert rel(dx, x.grad + dres + draw.float()) < 1e-5
    assert rel(dgamma, gamma.grad) < 1e-4
    # permuted destination rows (the logit-head gather): every other row dropped
    dest = torch.full((M,), -1, device=DEV, dtype=torch.int32)
    dest[::2] = torch.arange((M + 1) // 2, device=DEV, dtype=torch.int32).flip(0)
    y2 = torch.zeros((M + 1) // 2, D, device=DEV, dtype=ydt)
    lib.layernorm_fwd(x.detach(), gamma.detach(), y2, None, None, dest)
    assert torch.equal(y2[dest[::2].long()], y[::2])
    dx2 = torch.empty(M, D, device=DEV)
    dg2 = torch.zeros(D, device=DEV)
    dyp = torch.randn((M + 1) // 2, D, device=DEV).bfloat16()
    lib.layernorm_bwd(dyp, x.detach(), stats, gamma.detach(), dx2, dg2, src_row=dest)
    x.grad = None; gamma.grad = None
    full = torch.zeros(M, D, device=DEV)
    full[::2] = dyp[dest[::2].long()].float()
    F.layer_norm(x, (D,), gamma, None, 1e-5).backward(full)
    assert rel(dx2, x.grad) < 1e-5 and rel(dg2, gamma.grad) < 1e-4


@pytest.mark.parametrize("M,h", [(50, 2), (300, 8), (17, 3)])
def test_qk_l2norm(lib, M, h):
    torch.manual_seed(M)
    q = torch.randn(M, h * 64, device=DEV).bfloat16()
    kv = torch.randn(M, 128, device=DEV).bfloat16()
    qs = (1 + 0.3 * torch.randn(64, device=DEV)).requires_grad_(True)
    ks = (1 + 0.3 * torch.randn(64, device=DEV)).requires_grad_(True)
    qn = torch.empty_like(q); kvn = torch.empty_like(kv)
    lib.qk_l2norm_fwd(q, kv, qs.detach(), ks.detach(), qn, kvn, h)
    qf = q.float().requires_grad_(True); kvf = kv.float().requires_grad_(True)
    qr = F.normalize(qf.view(M, h, 64), dim=-1) * qs
    kr = F.normalize(kvf[:, :64], dim=-1) * ks
    assert rel(qn, qr.reshape(M, -1).detach()) < 4e-3
    assert rel(kvn[:, :64], kr.detach()) < 4e-3
    assert torch.equal(kvn[:, 64:], kv[:, 64:])
    dqn = torch.randn(M, h * 64, device=DEV); dkvn = torch.randn(M, 128, device=DEV)
    (qr.reshape(M, -1) * dqn).sum().backward(retain_graph=True)
    (kr * dkvn[:, :64]).sum().backward()
    dq = torch.empty_like(q); dkv = torch.empty_like(kv)
    dqs = torch.zeros(64, device=DEV); dks = torch.zeros(64, device=DEV)
    lib.qk_l2norm_bwd(dqn, dkvn, q, kv, qs.detach(), ks.detach(), dq, dkv, dqs, dks, h)
    assert rel(dq, qf.grad) < 4e-3
    assert rel(dkv[:, :64], kvf.grad[:, :64]) < 4e-3
    assert rel(dkv[:, 64:], dkvn[:, 64:]) < 4e-3
    assert rel(dqs, qs.grad) < 1e-4 and rel(dks, ks.grad) < 1e-4


def test_sgemm_small_and_silu(lib):
    torch.manual_seed(3)
    A = torch.randn(300, 70, device=DEV); W = torch.randn(90, 70, device=DEV); b = torch.randn(90, device=DEV)
    C = torch.empty(300, 90, device=DEV); Z = torch.empty_like(C)
    lib.sgemm_small(A, (70, 1), W, (1, 70), C, (90, 1), 300, 90, 70, Z=Z, bias=b, act=1)
    z = A @ W.t() + b
    assert rel(Z, z) < 1e-5 and rel(C, F.silu(z)) < 1e-5
    # transposed output + accumulate, A^T B form
    Ct = torch.ones(90, 300, device=DEV)
    lib.sgemm_small(A, (70, 1), W, (1, 70), Ct, (1, 300), 300, 90, 70, accumulate=True)
    assert rel(Ct, (A @ W.t()).t() + 1) < 1e-5
    dW = torch.empty(90, 70, device=DEV)
    dZ = torch.randn(300, 90, device=DEV)
    lib.sgemm_small(dZ, (1, 90), A, (70, 1), dW, (70, 1), 90, 70, 300)
    assert rel(dW, dZ.t() @ A) < 1e-5
    zz = z.clone().requires_grad_(True)
    F.silu(zz).backward(dZ)
    out = torch.empty_like(dZ)
    out_bf = torch.full_like(dZ, float("nan"), dtype=torch.bfloat16)
    lib.silu_bwd(dZ, z.contiguous(), out, out_bf)
    assert rel(out, zz.grad) < 1e-5
    assert torch.equal(out_bf, out.bfloat16())
    cs = torch.empty(90, device=DEV)
    lib.colsum(dZ, 90, 1, cs, 300, 90)
    assert rel(cs, dZ.sum(0)) < 1e-5
    cs0 = torch.randn(90, device=DEV)
    cs = cs0.clone()
    lib.colsum(dZ, 90, 1, cs, 300, 90, accumulate=True)
    assert rel(cs, cs0.double() + dZ.double().sum(0)) < 1e-6
    # split-K path (accumulate, no activation, no Z, K >= 128, < 64 output tiles): each K slice adds its partial
    # product into C atomically and only slice 0 adds the bias.  The rel-pos weight-gradient shapes dW4 [h, Hr] =
    # dY^T a3 and dW0 [Hr, 1] = dz^T x, on top of a non-zero C, against fp64
    for K in (128, 1000, 2048):
        for form in ("dW4", "dW0"):
            if form == "dW4":
                M, N_ = 8, 512
                dT = torch.randn(M, K, device=DEV)               # [h, N]
                a = torch.randn(K, N_, device=DEV)               # [N, Hr]
                args = (dT, (K, 1), a, (N_, 1))
                ref = dT.double() @ a.double()
            else:
                M, N_ = 512, 1
                dz = torch.randn(K, M, device=DEV)               # [N, Hr], read transposed
                x = torch.arange(K, device=DEV, dtype=torch.float32)[:, None] / K
                args = (dz, (1, M), x, (1, 1))
                ref = dz.double().t() @ x.double()
            C0 = torch.randn(M, N_, device=DEV) * float(ref.std())
            for bias in (None, torch.randn(N_, device=DEV) * float(ref.std())):
                C = C0.clone()
                lib.sgemm_small(*args, C, (N_, 1), M, N_, K, bias=bias, accumulate=True)
                want = ref + C0.double() + (bias.double()[None] if bias is not None else 0)
                assert rel(C, want) < 1e-5, (K, form, bias is not None, rel(C, want))


def test_split3_bias_silu_arange(lib):
    """The fp32 -> bf16x3 split (bit-exact, both layouts, strided source, grid-stride loop run more than once at the
    real size N=2048 x Hr=512), the fused bias + SiLU of the hidden layers and the distance ramp."""
    torch.manual_seed(11)
    R_, C_ = 2048, 512
    big = torch.randn(R_, C_ + 40, device=DEV) * torch.exp(2 * torch.randn(R_, C_ + 40, device=DEV))
    big[0, :4] = torch.tensor([0.0, -0.0, 1e-30, 3e38])
    for src in (big[:, :C_].contiguous(), big[:, 40:]):
        hi = src.bfloat16()
        lo = (src - hi.float()).bfloat16()
        for weight_mode, order in ((False, (hi, hi, lo)), (True, (hi, lo, hi))):
            dst = torch.full((R_, 3 * C_), float("nan"), device=DEV, dtype=torch.bfloat16)
            lib.split3_bf16(src, dst, weight_mode=weight_mode)
            for j, want in enumerate(order):
                assert torch.equal(dst[:, j * C_:(j + 1) * C_], want), (weight_mode, j)
    # the split is what the bf16x3 products rely on: hi + lo reproduces fp32 to ~2^-16 relative
    src = big[:, :C_]
    assert rel(src.bfloat16().double() + (src - src.bfloat16().float()).bfloat16().double(), src) < 2 ** -15
    z0 = torch.randn(R_, C_, device=DEV) * 4
    bias = torch.randn(C_, device=DEV)
    z = z0.clone()
    a = torch.full_like(z, float("nan"))
    lib.bias_silu(z, bias, a)
    assert torch.equal(z, z0 + bias)
    assert rel(a, F.silu(z.double())) < 1e-6
    for n in (75, 2048, 4097):
        out = torch.full((n, 1), float("nan"), device=DEV)
        lib.arange_f32(out)
        assert torch.equal(out[:, 0], torch.arange(n, device=DEV, dtype=torch.float32))


@pytest.mark.parametrize("Hr", [32, 64, 512])
@pytest.mark.parametrize("N", [75, 1021, 2048])
def test_bf16x3_gemm_accuracy(lib, Hr, N):
    """The three bf16x3 product forms of the rel-pos MLP (engine.py _relpos_table / _relpos_backward), fed by
    split3_bf16, against fp64 of the fp32 operands: forward A3 W3^T; dW += dz^T a over strided [:, :Hr] / [:, 2Hr:]
    column views with the output as addend; da = dz W in three accumulating calls.  Each must be fp32-class (rel-L2
    <= 5e-5) AND at least 50x more accurate than the plain bf16 product (hi x hi) of the same operands, which it is
    only if every lo term is present and in its column block.  Hr = 32 / 64: K below / at the GEMM's 64-wide k-block."""
    torch.manual_seed(Hr + N)
    a = F.silu(torch.randn(N, Hr, device=DEV) * 3)
    w = (torch.rand(Hr, Hr, device=DEV) * 2 - 1) / math.sqrt(Hr)
    dz = torch.randn(N, Hr, device=DEV)
    a3 = torch.empty(N, 3 * Hr, device=DEV, dtype=torch.bfloat16)
    w3 = torch.empty(Hr, 3 * Hr, device=DEV, dtype=torch.bfloat16)
    dz3 = torch.empty(N, 3 * Hr, device=DEV, dtype=torch.bfloat16)
    lib.split3_bf16(a, a3)
    lib.split3_bf16(w, w3, weight_mode=True)
    lib.split3_bf16(dz, dz3)
    a_hi, a_lo, dz_hi, dz_lo = a3[:, :Hr], a3[:, 2 * Hr:], dz3[:, :Hr], dz3[:, 2 * Hr:]
    w_hi, w_lo = w3[:, :Hr], w3[:, Hr:2 * Hr]
    errs = {}
    # forward: z = A3 . W3^T (K = 3 Hr), fp32 out
    ref = a.double() @ w.double().t()
    z3 = torch.full((N, Hr), float("nan"), device=DEV)
    z1 = torch.full((N, Hr), float("nan"), device=DEV)
    lib.gemm(a3, w3, z3, block_n=128)
    lib.gemm(a_hi, w_hi, z1, block_n=128)
    errs["fwd"] = (rel(z3, ref), rel(z1, ref))
    # dW += dz^T a: both operands MN-major, three accumulating products onto a non-zero gradient
    prod = dz.double().t() @ a.double()
    g0 = torch.randn(Hr, Hr, device=DEV) * float(prod.std())
    gw3, gw1 = g0.clone(), g0.clone()
    for x, y in ((dz_hi, a_hi), (dz_hi, a_lo), (dz_lo, a_hi)):
        lib.gemm(x, y, gw3, a_mn=True, b_mn=True, M=Hr, N=Hr, K=N, addend=gw3, block_n=128)
    lib.gemm(dz_hi, a_hi, gw1, a_mn=True, b_mn=True, M=Hr, N=Hr, K=N, addend=gw1, block_n=128)
    nrm = float(prod.norm())
    errs["dW"] = (float((gw3.double() - g0.double() - prod).norm()) / nrm, float((gw1.double() - g0.double() - prod).norm()) / nrm)
    # da = dz W: B MN-major, three calls, the last two accumulating
    ref = dz.double() @ w.double()
    da3 = torch.full((N, Hr), float("nan"), device=DEV)
    da1 = torch.full((N, Hr), float("nan"), device=DEV)
    lib.gemm(dz_hi, w_hi, da3, b_mn=True, M=N, N=Hr, K=Hr, block_n=128)
    lib.gemm(dz_hi, w_lo, da3, b_mn=True, M=N, N=Hr, K=Hr, addend=da3, block_n=128)
    lib.gemm(dz_lo, w_hi, da3, b_mn=True, M=N, N=Hr, K=Hr, addend=da3, block_n=128)
    lib.gemm(dz_hi, w_hi, da1, b_mn=True, M=N, N=Hr, K=Hr, block_n=128)
    errs["da"] = (rel(da3, ref), rel(da1, ref))
    print(f"bf16x3 Hr={Hr} N={N}: " + "  ".join(f"{k} {e3:.2e} (bf16 {e1:.2e})" for k, (e3, e1) in errs.items()))
    for k, (e3, e1) in errs.items():
        assert e3 <= 5e-5 and e3 * 50 <= e1, (k, e3, e1)


# ------------------------------------------------------------------------------------------------ attention
def _attn_ref(qn, kvn, table, key_mask, B, N, h, scale=8.0):
    q = qn.float().view(B, N, h, 64).permute(0, 2, 1, 3)
    k = kvn.float()[..., :64].view(B, N, 64)
    v = kvn.float()[..., 64:].view(B, N, 64)
    sim = torch.einsum("bhid,bjd->bhij", q, k) * scale
    i = torch.arange(N, device=qn.device)
    delta = i[:, None] - i[None, :]
    sim = sim + table[:, delta.clamp_min(0)][None]
    neg = -torch.finfo(torch.float32).max
    if key_mask is not None:
        sim = sim.masked_fill(~key_mask.bool()[:, None, None, :], neg)
    sim = sim.masked_fill((delta < 0)[None, None], neg)
    p = sim.softmax(-1)
    return torch.einsum("bhij,bjd->bhid", p, v).permute(0, 2, 1, 3).reshape(B, N, h * 64)


@pytest.mark.parametrize("B,N,h", [(2, 48, 2), (2, 200, 8), (1, 131, 3), (2, 300, 8), (1, 520, 16), (2, 1024, 8), (1, 1024, 16),
                                   (1, 2048, 8), (1, 700, 4)])
def test_attention_fwd_bwd(lib, B, N, h):
    torch.manual_seed(N + h)
    M = B * N
    qn = F.normalize(torch.randn(M, h, 64, device=DEV), dim=-1).reshape(M, h * 64).bfloat16()
    kv = torch.randn(M, 128, device=DEV)
    kv[:, :64] = F.normalize(kv[:, :64], dim=-1)
    kvn = kv.bfloat16()
    table = (torch.randn(h, 1, device=DEV) * 0.05 * torch.arange(N + 8, device=DEV)[None] + 0.3 * torch.randn(h, N + 8, device=DEV)).contiguous()
    key_mask = (torch.rand(B, N, device=DEV) > 0.2).to(torch.uint8)
    key_mask[:, 0] = 1
    out = torch.empty(M, h * 64, device=DEV, dtype=torch.bfloat16)
    lse2 = torch.empty(B, N * h, device=DEV)
    lib.attn_fwd(qn, kvn, table, key_mask, out, lse2, B, N, h)
    out_tc = torch.full((M, h * 64), float("nan"), device=DEV, dtype=torch.bfloat16)
    lse_tc = torch.full((B, N * h), float("nan"), device=DEV)
    lib.attn_fwd_tc(qn, kvn, table, key_mask, out_tc, lse_tc, B, N, h)
    torch.cuda.synchronize()
    assert rel(out_tc, out) < 6e-3, rel(out_tc, out)
    assert float((lse_tc - lse2).abs().max()) < 2e-2
    qf = qn.float().requires_grad_(True); kvf = kvn.float().requires_grad_(True); tf = table.clone().requires_grad_(True)
    ref = _attn_ref(qf, kvf, tf, key_mask, B, N, h)
    assert rel(out, ref.detach().reshape(M, -1)) < 6e-3
    d_o = torch.randn(M, h * 64, device=DEV).bfloat16()
    ref.backward(d_o.float().view(B, N, h * 64))
    dqn = torch.zeros(M, h * 64, device=DEV); dkvn = torch.zeros(M, 128, device=DEV)
    dtab = torch.zeros_like(table)
    dsum = torch.empty(M * h, device=DEV)
    lib.attn_bwd(qn, kvn, d_o, out, lse2, table, key_mask, dsum, dqn, dkvn, dtab, B, N, h)
    assert rel(dqn, qf.grad) < 1.5e-2
    assert rel(dkvn, kvf.grad) < 1.5e-2
    assert rel(dtab[:, :N], tf.grad[:, :N]) < 1.5e-2
    # tcgen05 backward
    # dqn / dkvn are overwritten (cleared inside the call): poison them to pin that contract; dtable accumulates
    dqn2 = torch.full((M, h * 64), float("nan"), device=DEV); dkvn2 = torch.full((M, 128), float("nan"), device=DEV); dtab2 = torch.zeros_like(table)
    lib.attn_bwd_tc(qn, kvn, d_o, out, lse2, table, key_mask, dsum, dqn2, dkvn2, dtab2, B, N, h)
    torch.cuda.synchronize()
    assert rel(dqn2, qf.grad) < 1.5e-2, rel(dqn2, qf.grad)
    assert rel(dkvn2, kvf.grad) < 1.5e-2, rel(dkvn2, kvf.grad)
    # bias gradient: diagonal sums of the hi/lo-split (fp32-class) dS inside the kernel
    assert rel(dtab2[:, :N], tf.grad[:, :N]) < 1.5e-2, rel(dtab2[:, :N], tf.grad[:, :N])
    assert float(dtab2[:, N:].abs().max()) == 0.0
    print(f"attn bwd B={B} N={N} h={h}: dq {rel(dqn2, qf.grad):.2e} dkv {rel(dkvn2, kvf.grad):.2e} dtable tc {rel(dtab2[:, :N], tf.grad[:, :N]):.2e} "
          f"(mma.sync {rel(dtab[:, :N], tf.grad[:, :N]):.2e})")


# ------------------------------------------------------------------------------------------------ conv-GEGLU feed-forward middle
def _ileave_cols(F_, Fp):
    """canonical column (value c | gate F+c) -> column of the interleaved [M, 2Fp] layout."""
    c = torch.arange(F_)
    a = (c // 128) * 256 + (c % 128)
    return torch.cat([a, a + 128])


@pytest.mark.parametrize("B,N,d,F_", [(2, 37, 64, 170), (2, 130, 128, 341), (1, 300, 1024, 2730)])
@pytest.mark.parametrize("drop_p", [0.0, 0.1])
@pytest.mark.parametrize("adt", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
def test_ffn_up_fused_and_mid_bwd(lib, B, N, d, F_, drop_p, adt):
    """gemm_ffn_up (GEMM + conv + GEGLU + row sums in the epilogue) + ffn_norm_fwd + ffn_mid_bwd vs torch, with the
    forward activations / weights in bf16 and in fp16 (gradients are bf16 in both)."""
    torch.manual_seed(F_)
    Fp = (F_ + 127) // 128 * 128
    M = B * N
    xn = torch.randn(M, d, device=DEV).to(adt)
    W1 = ((torch.rand(2 * F_, d, device=DEV) * 2 - 1) / math.sqrt(d))
    cw = (torch.rand(2 * F_, 3, device=DEV) * 2 - 1) / math.sqrt(3)
    gam = 1 + 0.2 * torch.randn(F_, device=DEV)
    w1p = torch.empty(2 * Fp, d, device=DEV, dtype=adt)
    cwp = torch.empty(2 * Fp, 3, device=DEV); gp = torch.empty(Fp, device=DEV)
    lib.pack(W1, d, 2 * F_, d, w1p, 2 * Fp, d, split_dst=-1, split_src=F_)
    lib.pack(cw, 3, 2 * F_, 3, cwp, 2 * Fp, 3, split_dst=-1, split_src=F_)
    lib.pack(gam, F_, 1, F_, gp, 1, Fp)
    cols = _ileave_cols(F_, Fp).to(DEV)
    assert torch.equal(w1p[cols], W1.to(adt)) and torch.equal(cwp[cols], cw)
    u = torch.full((M, 2 * Fp), float("nan"), device=DEV, dtype=adt)
    h = torch.full((M, Fp), float("nan"), device=DEV, dtype=adt)
    rowsum = torch.full((M, Fp // 128, 2), float("nan"), device=DEV)
    lib.gemm_ffn_up(xn, w1p, cwp, u, h, rowsum, N, Fp)
    hn = torch.empty(M, Fp, device=DEV, dtype=adt); stats = torch.empty(M, 2, device=DEV)
    seed = torch.tensor([99], dtype=torch.int64, device=DEV)
    kbits = torch.zeros(M, Fp // 8, device=DEV, dtype=torch.uint8)
    hn_b = torch.empty(M, Fp, device=DEV, dtype=torch.bfloat16) if adt == torch.float16 else hn    # what the backward pass reads
    lib.ffn_norm_fwd(h, rowsum, gp, hn, stats, F_, Fp, drop_p, seed, 3, keep_bits=kbits if drop_p > 0 else None,
                     hn_copy=hn_b if adt == torch.float16 else None)
    torch.cuda.synchronize()
    assert rel(hn_b, hn) < 4e-3
    # reference (the conv sees the bf16-rounded u, as in the unfused formulation)
    u_ref = (xn.float() @ W1.to(adt).float().t())
    assert rel(u[:, cols], u_ref) < 5e-3
    uf = u[:, cols].float().requires_grad_(True); cwr = cw.clone().requires_grad_(True); gr = gam.clone().requires_grad_(True)
    ub = uf.view(B, N, 2 * F_)
    up = F.pad(ub, (0, 0, 2, 0))
    y = up[:, 0:-2] * cwr[:, 0] + up[:, 1:-1] * cwr[:, 1] + up[:, 2:] * cwr[:, 2]
    hmid = F.gelu(y[..., F_:]) * y[..., :F_]
    assert rel(h[:, :F_], hmid.detach().reshape(M, F_)) < 5e-3
    assert float(h[:, F_:].abs().max()) == 0
    assert rel(rowsum.sum(1)[:, 0], hmid.detach().reshape(M, F_).sum(1)) < 2e-3
    ref = F.layer_norm(hmid, (F_,), gr, None, 1e-5).reshape(M, F_)
    if drop_p > 0:
        keep = ((kbits[:, :, None] >> torch.arange(8, device=DEV, dtype=torch.uint8)) & 1).bool().reshape(M, Fp)[:, :F_]
        assert torch.equal(keep | (ref.detach().abs() < 1e-3), (hn[:, :F_] != 0) | (ref.detach().abs() < 1e-3))
        assert abs(1 - keep.float().mean().item() - drop_p) < 0.02
        ref = ref * keep / (1 - drop_p)
    assert float(hn[:, F_:].abs().max()) == 0
    assert rel(hn[:, :F_], ref.detach()) < 8e-3
    # backward
    dhn = torch.zeros(M, Fp, device=DEV, dtype=torch.bfloat16)
    dhn[:, :F_] = torch.randn(M, F_, device=DEV).bfloat16()
    ref.backward(dhn[:, :F_].float())
    du = torch.empty(M, 2 * Fp, device=DEV, dtype=torch.bfloat16); rowstat = torch.empty(M, 2, device=DEV)
    # parameter gradients are accumulated (+=) in the parameters' own layouts: start from a known non-zero value
    dg = torch.full((F_,), 0.5, device=DEV); dcw = torch.full((2 * F_, 3), -0.25, device=DEV)
    lib.ffn_mid_bwd(dhn, hn_b, u, stats, cwp, gp, rowstat, du, dg, dcw, B, N, F_, Fp, drop_p, keep_bits=kbits if drop_p > 0 else None)
    assert rel(du[:, cols], uf.grad) < 1.5e-2
    assert rel(dg - 0.5, gr.grad) < 8e-3
    assert rel(dcw + 0.25, cwr.grad) < 1.5e-2
    if Fp % 256 == 0:
        # the same backward with the row sums taken in the epilogue of the GEMM that produces dhn (omlm_gemm16_rowstat):
        # dhn = dx W2 for a random dx; partial sums per 128-column half tile against fp32 torch
        dx = torch.randn(M, d, device=DEV).bfloat16()
        w2 = ((torch.rand(d, Fp, device=DEV) * 2 - 1) / math.sqrt(d)).bfloat16()
        w2[:, F_:] = 0
        dhn2 = torch.empty(M, Fp, device=DEV, dtype=torch.bfloat16)
        part = torch.full((M, Fp // 128, 2), float("nan"), device=DEV)
        ks = 1.0 / (1.0 - drop_p) if drop_p > 0 else 1.0
        lib.gemm_rowstat(dx, w2, dhn2, hn_b, gp, part, b_mn=True, M=M, N=Fp, K=d, keep_bits=kbits if drop_p > 0 else None, keep_scale=ks)
        dref = dx.float() @ w2.float()
        assert rel(dhn2, dref) < 4e-3
        keep_f = ((kbits[:, :, None] >> torch.arange(8, device=DEV, dtype=torch.uint8)) & 1).float().reshape(M, Fp) if drop_p > 0 else torch.ones(M, Fp, device=DEV)
        s1 = (gp[None] * keep_f * ks * dref).view(M, Fp // 128, 128).sum(-1)
        s2 = (dref * hn_b.float()).view(M, Fp // 128, 128).sum(-1)
        assert rel(part[..., 0], s1) < 2e-3 and rel(part[..., 1], s2) < 2e-3, (rel(part[..., 0], s1), rel(part[..., 1], s2))
        # ... and the tile kernel fed with those partial sums equals the tile kernel with its own statistics pass
        du_a = torch.empty_like(du); du_b = torch.empty_like(du)
        dga = torch.zeros(F_, device=DEV); dgb = torch.zeros(F_, device=DEV); dca = torch.zeros(2 * F_, 3, device=DEV); dcb = torch.zeros(2 * F_, 3, device=DEV)
        kb = kbits if drop_p > 0 else None
        lib.ffn_mid_bwd(dhn2, hn_b, u, stats, cwp, gp, part, du_a, dga, dca, B, N, F_, Fp, drop_p, keep_bits=kb, rowstat_parts=Fp // 128)
        lib.ffn_mid_bwd(dhn2, hn_b, u, stats, cwp, gp, rowstat, du_b, dgb, dcb, B, N, F_, Fp, drop_p, keep_bits=kb)
        assert rel(du_a, du_b) < 3e-3 and rel(dga, dgb) < 3e-3 and rel(dca, dcb) < 3e-3, (rel(du_a, du_b), rel(dga, dgb), rel(dca, dcb))


# ------------------------------------------------------------------------------------------------ loss / optimiser
def test_cross_entropy(lib):
    torch.manual_seed(0)
    rows, C, Cp = 333, 1025, 1088
    logits = (torch.randn(rows, C, device=DEV) * 8).requires_grad_(True)
    labels = torch.randint(0, C, (rows,), device=DEV, dtype=torch.int32)
    labels[5] = -100
    acc = torch.zeros(2, device=DEV)
    dl = torch.full((rows, Cp), 7.0, device=DEV, dtype=torch.bfloat16)
    lib.cross_entropy(logits.detach(), labels, C, acc, grad_scale=0.37, dlogits=dl)
    ref = F.cross_entropy(logits, labels.long(), ignore_index=-100, reduction="sum")
    assert abs(float(acc[0]) - float(ref)) / float(ref) < 1e-5 and float(acc[1]) == rows - 1
    (ref * 0.37).backward()
    assert rel(dl[:, :C], logits.grad) < 4e-3
    assert float(dl[:, C:].abs().max()) == 0
    # strided label view of a logit-head group: rows ordered (sequence b, step t), labels at plane[b, off + qi + q t];
    # the weighted loss goes straight into the accumulator
    B, cnt, q, qi, off = 9, 37, 3, 1, 5
    plane = torch.randint(0, C, (B, off + q * cnt + 2), device=DEV, dtype=torch.int32)
    lg = torch.randn(B * cnt, C, device=DEV) * 4
    acc2 = torch.zeros(2, device=DEV)
    lib.cross_entropy(lg, plane[0, off + qi:], C, acc2, rows=B * cnt, label_stride=q, rows_per_batch=cnt, batch_stride=plane.stride(0), loss_scale=0.25)
    lab = plane[:, off + qi::q][:, :cnt].reshape(-1).long()
    ref2 = 0.25 * F.cross_entropy(lg, lab, reduction="sum")
    assert abs(float(acc2[0]) - float(ref2)) / float(ref2) < 1e-5 and float(acc2[1]) == B * cnt


def test_adamw_matches_torch(lib):
    torch.manual_seed(0)
    n_decay, n = 5000, 7003
    p0 = torch.randn(n, device=DEV)
    pa = torch.nn.Parameter(p0[:n_decay].clone().view(50, 100)); pb = torch.nn.Parameter(p0[n_decay:].clone())
    opt = torch.optim.AdamW([{"params": [pa]}, {"params": [pb], "weight_decay": 0}], lr=3e-4, weight_decay=1e-2, betas=(0.9, 0.99), eps=1e-8)
    p = p0.clone(); m = torch.zeros(n, device=DEV); v = torch.zeros(n, device=DEV)
    for t in range(1, 4):
        g = torch.randn(n, device=DEV) * (0.01 if t == 2 else 1.0)
        pa.grad = g[:n_decay].clone().view(50, 100); pb.grad = g[n_decay:].clone()
        torch.nn.utils.clip_grad_norm_([pa, pb], 0.5)
        opt.step()
        acc = torch.zeros(1, device=DEV, dtype=torch.float64)
        lib.grad_sumsq(g, acc)
        assert abs(float(acc) - float((g.double() ** 2).sum())) / float((g.double() ** 2).sum()) < 1e-6
        hyper = torch.tensor([3e-4, 0.9, 0.99, 1e-8, 1e-2, 1 - 0.9 ** t, 1 - 0.99 ** t, 0.5, 1.0], device=DEV)
        lib.adamw_step(p, g, m, v, n_decay, hyper, acc)
        ref = torch.cat([pa.detach().reshape(-1), pb.detach()])
        assert rel(p, ref) < 1e-6


def test_attention_fwd_speed(lib):
    """Prints the two forward attention paths side by side at the cfg2 shape (not a benchmark)."""
    B, N, h = 16, 1024, 8
    M = B * N
    torch.manual_seed(0)
    qn = F.normalize(torch.randn(M, h, 64, device=DEV), dim=-1).reshape(M, h * 64).bfloat16()
    kvn = torch.randn(M, 128, device=DEV).bfloat16()
    table = (torch.randn(h, 1, device=DEV) * 0.05 * torch.arange(N, device=DEV)[None]).contiguous()
    key_mask = (torch.rand(B, N, device=DEV) > 0.15).to(torch.uint8); key_mask[:, 0] = 1
    out = torch.empty(M, h * 64, device=DEV, dtype=torch.bfloat16); lse2 = torch.empty(B, N * h, device=DEV)
    for name, fn in (("mma.sync", lib.attn_fwd), ("tcgen05", lib.attn_fwd_tc)):
        for _ in range(3):
            fn(qn, kvn, table, key_mask, out, lse2, B, N, h)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            fn(qn, kvn, table, key_mask, out, lse2, B, N, h)
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 10
        print(f"attn fwd {name}: {ms:.3f} ms  {B * N * h * 64 * (N + 1) * 2 / ms / 1e9:.0f} TFLOP/s (causal flops)")
