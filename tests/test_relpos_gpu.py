"""The relative-position bias of the engine against fp64, stage by stage: the table the forward pass builds
(Engine.build_bias_table), the MLP backward given an exact table gradient (Engine.bias_table_backward), and the
attribution of the end-to-end rel-pos gradient error to the attention backward's d(table) rather than the MLP.

The fp64 reference is oracle.restatement.rel_pos_table (autograd for the gradients) on the engine's own fp32
parameters.  One-layer semantic models; the workspace of batch 1 with sequences [12, N - 14] has exactly N positions."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda"
RP = "transformer.rel_pos_bias."
SHAPES = [(64, 2, 75), (1024, 8, 1024), (1024, 16, 2048)]       # (d, h, N): d = 64 gives Hr = 32 < the GEMM k-block

# bounds from a B200 run (1000 W power limit) with ~1.5x margin; the tests print the measured errors
TABLE_REL, TABLE_MAX = 1.5e-5, 2.5e-5     # table rel-L2 (measured <= 8.6e-6), max |diff| / max |table| (<= 1.6e-5)
MLP_BWD_RANDOM = 1.5e-4                   # rel-L2 of every rel-pos gradient, random d(table) (<= 9.2e-5, at N = 2048)
MLP_BWD_ZERO_SUM = 1.2e-3                 # the same, zero-sum-per-head d(table) like attention's (<= 7.5e-4)
NET3_BIAS_ZERO_SUM = 2e-8                 # |net.3.bias grad - ref| / |net.3.weight grad| for that d(table) (<= 9.4e-9)


def rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


@pytest.fixture(scope="module")
def lib():
    from open_musiclm_b200 import lib as L
    L.device_check()
    return L


def make_engine(d, h, N, bias_type="continuous"):
    import open_musiclm_b200 as O
    torch.manual_seed(d + h + N)
    m = O.create_semantic_transformer(dim=d, depth=1, heads=h, attn_dropout=0.0, ff_dropout=0.0,
                                      relative_position_bias_type=bias_type)
    eng = m.cuda().engine
    ws = eng.workspace(eng.plan(1, [12, N - 14]), True)
    assert ws["table"].shape == (h, N)
    eng.refresh_packed(force=True)
    return m, eng, ws


def rp_params(eng, dtype=torch.float64, grad=False):
    return {k: v.detach().to(dtype).requires_grad_(grad) for k, v in eng.pview.items() if k.startswith(RP)}


def table64(eng, N):
    from oracle import restatement as R
    return R.rel_pos_table(rp_params(eng), N, eng.bias_type, eng.h, dtype=torch.float64).to(DEV)


def ref_grads(eng, N, dT):
    """fp64 autograd of rel_pos_table(...).backward(dT) on the engine's parameters."""
    from oracle import restatement as R
    sd = rp_params(eng, grad=True)
    R.rel_pos_table(sd, N, eng.bias_type, eng.h, dtype=torch.float64).backward(dT.double().to(DEV))
    return {k: v.grad for k, v in sd.items()}


def kernel_grads(eng, ws, N, dT):
    """Engine.bias_table_backward on d(table) = dT (needs the forward's saved activations: build_bias_table first)."""
    ws["dtable"].copy_(dT)
    eng.arena_g.zero_()
    eng.bias_table_backward(ws, N)
    out = {k: v.clone() for k, v in eng.gview.items() if k.startswith(RP)}
    untouched = eng.arena_g.clone()
    for k in out:
        o = eng.layout[k]
        untouched[o:o + out[k].numel()] = 0
    assert float(untouched.abs().max()) == 0.0          # nothing outside the rel-pos gradients is written
    eng.arena_g.zero_()
    return out


# ------------------------------------------------------------------------------------------------ forward table
@pytest.mark.parametrize("scaled", [False, True], ids=["init", "max100"])
@pytest.mark.parametrize("d,h,N", SHAPES)
def test_continuous_table_vs_fp64(lib, d, h, N, scaled):
    """The table from the SIMT first / last layers and the bf16x3 tcgen05 hidden layers is fp32-class, with the init
    weights and with the last layer scaled so that max |table| = 100 (the magnitude trained models reach)."""
    m, eng, ws = make_engine(d, h, N)
    if scaled:
        s = 100.0 / float(table64(eng, N).abs().max())
        eng.pview[RP + "net.3.weight"].mul_(s)
        eng.pview[RP + "net.3.bias"].mul_(s)
    ref = table64(eng, N)
    ws["table"].fill_(float("nan"))
    eng.build_bias_table(ws, N)
    got = ws["table"]
    r = rel(got, ref)
    mx = float((got.double() - ref).abs().max() / ref.abs().max())
    print(f"table d={d} h={h} N={N} {'max100' if scaled else 'init'}: max|table| {float(ref.abs().max()):.3g} "
          f"rel-L2 {r:.2e} max|diff|/max|table| {mx:.2e}")
    assert r <= TABLE_REL and mx <= TABLE_MAX, (r, mx)


@pytest.mark.parametrize("d,h,N", [(64, 2, 75), (64, 16, 2048)])
def test_t5_and_none_table_and_backward(lib, d, h, N):
    """t5: every causal distance falls into bucket 0, so the table is row 0 of the bucket embedding (exactly) and the
    gradient lands in bucket row 0 through colsum.  'none': a zero table and no gradient."""
    m, eng, ws = make_engine(d, h, N, "t5")
    eng.build_bias_table(ws, N)
    assert torch.equal(ws["table"].double(), table64(eng, N))
    dT = torch.randn(h, N, device=DEV)
    got = kernel_grads(eng, ws, N, dT)
    ref = ref_grads(eng, N, dT)
    k = RP + "relative_attention_bias.weight"
    assert float(ref[k][1:].abs().max()) == 0.0 and float(got[k][1:].abs().max()) == 0.0
    assert rel(got[k][0], ref[k][0]) < 1e-5, rel(got[k][0], ref[k][0])
    m, eng, ws = make_engine(d, h, N, "none")
    eng.build_bias_table(ws, N)
    assert float(ws["table"].abs().max()) == 0.0
    assert kernel_grads(eng, ws, N, dT) == {}


# ------------------------------------------------------------------------------------------------ MLP backward
@pytest.mark.parametrize("zero_sum", [False, True], ids=["random", "zero_sum"])
@pytest.mark.parametrize("d,h,N", SHAPES)
def test_mlp_backward_exact_input(lib, d, h, N, zero_sum):
    """bias_table_backward given an exact d(table), every rel-pos gradient against fp64 autograd.  With a zero-sum
    d(table) per head (attention's: sum_j dS_ij = 0) net.3.bias is analytically zero and is checked in absolute terms,
    against the scale of the net.3.weight gradient, as the parity tests do."""
    m, eng, ws = make_engine(d, h, N)
    eng.build_bias_table(ws, N)
    g = torch.Generator(device=DEV).manual_seed(N + h)
    dT = torch.randn(h, N, device=DEV, generator=g)
    if zero_sum:
        dT = dT - dT.mean(1, keepdim=True)
    got, ref = kernel_grads(eng, ws, N, dT), ref_grads(eng, N, dT)
    errs = {}
    for k in ref:
        if zero_sum and k.endswith("net.3.bias"):
            errs[k] = float((got[k].double() - ref[k]).norm() / ref[RP + "net.3.weight"].norm())
        else:
            errs[k] = rel(got[k], ref[k])
    print(f"MLP backward d={d} h={h} N={N} {'zero-sum' if zero_sum else 'random'} dT: " +
          " ".join(f"{k[len(RP) + 4:]} {e:.2e}" for k, e in errs.items()))
    for k, e in errs.items():
        bound = NET3_BIAS_ZERO_SUM if zero_sum and k.endswith("net.3.bias") else (MLP_BWD_ZERO_SUM if zero_sum else MLP_BWD_RANDOM)
        assert e <= bound, (k, e, bound)


# ------------------------------------------------------------------------------------------------ attribution
def _attn64(qn, kvn, table, key_mask, B, N, h, scale=8.0):
    """Causal cosine-sim MQA with the bias table (as the attention kernels compute it) in fp64."""
    q = qn.double().view(B, N, h, 64).permute(0, 2, 1, 3)
    k = kvn.double()[..., :64].view(B, N, 64)
    v = kvn.double()[..., 64:].view(B, N, 64)
    sim = torch.einsum("bhid,bjd->bhij", q, k) * scale
    i = torch.arange(N, device=qn.device)
    delta = i[:, None] - i[None, :]
    sim = sim + table[:, delta.clamp_min(0)][None]
    sim = sim.masked_fill(~key_mask.bool()[:, None, None, :], float("-inf"))
    sim = sim.masked_fill((delta < 0)[None, None], float("-inf"))
    return torch.einsum("bhij,bjd->bhid", sim.softmax(-1), v).permute(0, 2, 1, 3).reshape(B * N, h * 64)


@pytest.mark.parametrize("d,h,N,B", [(1024, 8, 1024, 2), (1024, 16, 2048, 1)])
def test_relpos_gradient_error_comes_from_attention_dtable(lib, d, h, N, B):
    """The rel-pos MLP gradients at N = 1024 / 2048 are further from fp64 than the 2e-2 met elsewhere.  Split the
    chain: the attention backward's d(table) (tcgen05 kernel, bf16 operands) against fp64 autograd of the same
    bf16 inputs, then the MLP backward fed with each.  MLP_bwd(exact d(table)) must be >= 20x closer to the fp64 chain
    than MLP_bwd(kernel d(table)): the error is the attention's, amplified by the cancelling diagonal sums."""
    m, eng, ws = make_engine(d, h, N)
    eng.build_bias_table(ws, N)
    table = ws["table"]
    torch.manual_seed(N + h)
    M = B * N
    qn = F.normalize(torch.randn(M, h, 64, device=DEV), dim=-1).reshape(M, h * 64).bfloat16()
    kv = torch.randn(M, 128, device=DEV)
    kv[:, :64] = F.normalize(kv[:, :64], dim=-1)
    kvn = kv.bfloat16()
    key_mask = (torch.rand(B, N, device=DEV) > 0.2).to(torch.uint8)
    key_mask[:, 0] = 1
    out = torch.empty(M, h * 64, device=DEV, dtype=torch.bfloat16)
    lse = torch.empty(B, N * h, device=DEV)
    lib.attn_fwd_tc(qn, kvn, table, key_mask, out, lse, B, N, h)
    d_o = torch.randn(M, h * 64, device=DEV).bfloat16()
    dqn = torch.empty(M, h * 64, device=DEV); dkvn = torch.empty(M, 128, device=DEV); dsum = torch.empty(M * h, device=DEV)
    dT_kernel = torch.zeros(h, N, device=DEV)
    lib.attn_bwd_tc(qn, kvn, d_o, out, lse, table, key_mask, dsum, dqn, dkvn, dT_kernel, B, N, h)
    t64 = table.double().clone().requires_grad_(True)
    _attn64(qn, kvn, t64, key_mask, B, N, h).backward(d_o.double())
    dT64 = t64.grad
    ref = ref_grads(eng, N, dT64)
    exact = kernel_grads(eng, ws, N, dT64.float())
    kern = kernel_grads(eng, ws, N, dT_kernel)
    print(f"attribution d={d} h={h} N={N} B={B}: d(table) rel-L2 {rel(dT_kernel, dT64):.2e}")
    for k in ref:
        if k.endswith("net.3.bias"):
            continue                                       # analytically zero for a zero-sum d(table)
        e_mlp, e_kern = rel(exact[k], ref[k]), rel(kern[k], ref[k])
        print(f"  {k[len(RP):]}: MLP_bwd(fp64 dT) {e_mlp:.2e}  MLP_bwd(kernel dT) {e_kern:.2e}  ratio {e_kern / max(e_mlp, 1e-30):.0f}")
        assert e_mlp * 20 <= e_kern, (k, e_mlp, e_kern)
