"""ORACLE — test infrastructure only.  Never imported by the product path.

CPU restatement (numpy for the integer/byte path, plain torch fp32 for the floating-point path) of
the reference's TokenConditionedTransformer training path.  It is written from the reference's
behaviour, function by function, and every function cites the reference file:line it follows
(paths relative to /root/reference).  It is pinned against the real reference by
`oracle/make_golden.py` (run in the authoring container, where /root/reference is importable) and
the committed fixtures under tests/golden/ — see tests/test_oracle_cpu.py.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import it.

State is a flat dict {reference state_dict key: tensor}; hyper-parameters live in `Cfg`.
"""
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import math
import numpy as np
import torch
import torch.nn.functional as F


@dataclass
class SeqInfo:
    """open_musiclm/open_musiclm.py:23-30 (TokenSequenceInfo)."""
    codebook_size: int
    num_quantizers: int


@dataclass
class Cfg:
    seqs: List[SeqInfo]
    dim: int
    depth: int
    heads: int
    dim_head: int = 64                      # transformer.py:172
    attn_scale: float = 8.0                 # transformer.py:178
    ff_dropout: float = 0.1
    grad_shrink_alpha: float = 0.1          # transformer.py:350, utils.py:60-61
    ce_weights: Optional[List[float]] = None
    mask_prob: float = 0.15                 # open_musiclm.py:228
    pad_id: int = -1
    use_conv_ff: bool = True                # transformer.py:349, 380: ConvFeedForward vs FeedForward
    rel_pos_bias_type: str = "continuous"   # transformer.py:353, 366-373: 'continuous' | 't5' | 'none'
    abs_pos: bool = False                   # open_musiclm.py:53-54, 81-82, 134-136: per-sequence absolute position embeddings
    max_abs_pos: int = 262

    @property
    def ff_inner(self) -> int:
        if not self.use_conv_ff:
            return int(self.dim * 4)        # transformer.py:153
        return int(self.dim * 2 * 4 / 3)    # transformer.py:141

    @property
    def ff_keys(self):
        """state_dict suffixes of the feed-forward Sequential: (pre-norm gamma, up weight, conv weight or None, inner gamma, down weight)."""
        if self.use_conv_ff:
            return ("0.gamma", "1.weight", "2.ds_conv.weight", "4.gamma", "6.weight")     # transformer.py:142-150
        return ("0.gamma", "1.weight", None, "3.gamma", "5.weight")                       # transformer.py:154-161


def semantic_cfg(dim=1024, depth=6, heads=8, codebook=1024, n_clap_q=12, **kw) -> Cfg:
    """open_musiclm.py:414-428 create_semantic_transformer."""
    return Cfg(seqs=[SeqInfo(codebook, n_clap_q), SeqInfo(codebook, 1)], dim=dim, depth=depth, heads=heads, **kw)


def coarse_cfg(dim=1024, depth=6, heads=8, codebook=1024, n_clap_q=12, n_coarse_q=3, **kw) -> Cfg:
    """open_musiclm.py:432-450 create_coarse_transformer."""
    return Cfg(seqs=[SeqInfo(codebook, n_clap_q), SeqInfo(codebook, 1), SeqInfo(codebook, n_coarse_q)],
               dim=dim, depth=depth, heads=heads, **kw)


def fine_cfg(dim=1024, depth=6, heads=8, codebook=1024, n_clap_q=12, n_coarse_q=3, n_fine_q=5, **kw) -> Cfg:
    """open_musiclm.py:454-472 create_fine_transformer."""
    return Cfg(seqs=[SeqInfo(codebook, n_clap_q), SeqInfo(codebook, n_coarse_q), SeqInfo(codebook, n_fine_q)],
               dim=dim, depth=depth, heads=heads, **kw)


# --------------------------------------------------------------------------------------------
# parameter initialisation with the reference's shapes / key names (values: reference defaults)
# --------------------------------------------------------------------------------------------

def init_state(cfg: Cfg, seed: int = 0) -> Dict[str, torch.Tensor]:
    """Shapes/keys of TokenConditionedTransformer.state_dict() (open_musiclm.py:66-94,
    transformer.py:24-31,39-53,122-150,195-212,364-383).  Distributions follow torch defaults
    (randn for start tokens / logit weights / embeddings, kaiming-uniform(a=sqrt(5)) for Linear and
    Conv1d); the RNG stream is NOT the reference's — parity tests load identical weights instead."""
    g = torch.Generator().manual_seed(seed)
    d, F_, h, dh = cfg.dim, cfg.ff_inner, cfg.heads, cfg.dim_head
    sd: Dict[str, torch.Tensor] = {}

    def lin(out_f, in_f):
        bound = 1.0 / math.sqrt(in_f)
        return (torch.rand(out_f, in_f, generator=g) * 2 - 1) * bound

    for i, s in enumerate(cfg.seqs):
        sd[f"start_tokens.{i}"] = torch.randn(d, generator=g)
        sd[f"logit_weights.{i}"] = torch.randn(s.num_quantizers, s.codebook_size + 1, d, generator=g)
        sd[f"embeddings.{i}.weight"] = torch.randn((s.codebook_size + 1) * s.num_quantizers, d, generator=g)
        if cfg.abs_pos:
            sd[f"absolute_position_embeddings.{i}.weight"] = torch.randn(cfg.max_abs_pos, d, generator=g)
    hid = d // 2                                    # transformer.py:367
    if cfg.rel_pos_bias_type == "continuous":
        sd["transformer.rel_pos_bias.net.0.0.weight"] = lin(hid, 1)
        sd["transformer.rel_pos_bias.net.0.0.bias"] = (torch.rand(hid, generator=g) * 2 - 1)
        for j in (1, 2):
            sd[f"transformer.rel_pos_bias.net.{j}.0.weight"] = lin(hid, hid)
            sd[f"transformer.rel_pos_bias.net.{j}.0.bias"] = (torch.rand(hid, generator=g) * 2 - 1) / math.sqrt(hid)
        sd["transformer.rel_pos_bias.net.3.weight"] = lin(h, hid)
        sd["transformer.rel_pos_bias.net.3.bias"] = (torch.rand(h, generator=g) * 2 - 1) / math.sqrt(hid)
    elif cfg.rel_pos_bias_type == "t5":
        sd["transformer.rel_pos_bias.relative_attention_bias.weight"] = torch.randn(32, h, generator=g)
    for l in range(cfg.depth):
        p = f"transformer.layers.{l}."
        sd[p + "0.q_scale"] = torch.ones(dh)
        sd[p + "0.k_scale"] = torch.ones(dh)
        sd[p + "0.norm.gamma"] = torch.ones(d)
        sd[p + "0.norm.beta"] = torch.zeros(d)
        sd[p + "0.to_q.weight"] = lin(h * dh, d)
        sd[p + "0.to_kv.weight"] = lin(2 * dh, d)
        sd[p + "0.to_out.0.weight"] = lin(d, h * dh)
        k_g1, k_w1, k_conv, k_gin, k_w2 = cfg.ff_keys
        sd[p + "2." + k_g1] = torch.ones(d)
        sd[p + "2." + k_g1.replace("gamma", "beta")] = torch.zeros(d)
        sd[p + "2." + k_w1] = lin(2 * F_, d)
        if k_conv is not None:
            sd[p + "2." + k_conv] = ((torch.rand(2 * F_, 1, 3, generator=g) * 2 - 1) / math.sqrt(3.0))
        sd[p + "2." + k_gin] = torch.ones(F_)
        sd[p + "2." + k_gin.replace("gamma", "beta")] = torch.zeros(F_)
        sd[p + "2." + k_w2] = lin(d, F_)
    sd["transformer.norm.gamma"] = torch.ones(d)
    sd["transformer.norm.beta"] = torch.zeros(d)
    return sd


# --------------------------------------------------------------------------------------------
# integer path (numpy, bit-exact contract)
# --------------------------------------------------------------------------------------------

def prepare_ids(cfg: Cfg, all_token_ids: Sequence[np.ndarray], return_loss: bool, forget_mask: Optional[np.ndarray] = None
                ) -> Tuple[List[np.ndarray], np.ndarray, Optional[List[np.ndarray]]]:
    """TokenConditionedTransformerWrapper.forward pre-processing, open_musiclm.py:336-376
    (+ append_eos_id, utils.py:112-117).  Returns (ids per sequence after eos append / last-token
    drop / in-place zeroing, key mask [B, N] bool, labels).  `forget_mask` is the [B, N] boolean
    keep-mask of generate_mask_with_prob (utils.py:49-56) when training, else None."""
    ids = [np.asarray(t).reshape(t.shape[0], -1).astype(np.int64) for t in all_token_ids]      # :340
    B = ids[0].shape[0]
    ids = [np.concatenate([t, np.full((B, 1), s.codebook_size, np.int64)], 1) for t, s in zip(ids, cfg.seqs)]  # :346-347
    labels = None
    if return_loss:
        labels = [t.copy() for t in ids]                                                        # :355
        ids[-1] = ids[-1][:, :-1]                                                               # :356
    masks = []
    for t, s in zip(ids[:-1], cfg.seqs[:-1]):
        m = (t != cfg.pad_id) & (t != s.codebook_size)                                          # :361
        t[~m] = 0                                                                               # :363 (in place)
        masks.append(np.concatenate([np.ones((B, 1), bool), m], 1))                             # :366
    masks.append(np.ones((B, ids[-1].shape[1] + 1), bool))                                      # :370-371
    mask = np.concatenate(masks, 1)
    if forget_mask is not None:
        mask = mask & forget_mask                                                               # :374-376
    return ids, mask, labels


def embedding_rows(cfg: Cfg, ids: Sequence[np.ndarray]) -> List[Tuple[np.ndarray, np.ndarray]]:
    """TokenConditionedTransformer.forward, open_musiclm.py:126-133 + get_embeds utils.py:126-143.
    Per sequence: (row index into embeddings[s].weight, pad flag).  Offsets use codebook_size (not
    codebook_size+1) and are added BEFORE the pad test."""
    out = []
    for t, s in zip(ids, cfg.seqs):
        c = t.copy()
        if s.num_quantizers > 1:
            c = c + (s.codebook_size * (np.arange(c.shape[1]) % s.num_quantizers))[None, :]     # :127-130
        pad = c == cfg.pad_id                                                                   # utils.py:133
        out.append((np.where(pad, 0, c), pad))                                                  # utils.py:134
    return out


def forgetful_mask(shape, mask_prob: float, rand: np.ndarray) -> np.ndarray:
    """generate_mask_with_prob, utils.py:49-56, given the randn draw `rand` [B, N]: the top
    int(N*p) positions per row (column 0 excluded) are dropped."""
    r = rand.astype(np.float32).copy()
    r[:, 0] = -np.finfo(np.float32).max
    n = shape[-1]
    k = min(int(n * mask_prob), n - 1)
    idx = np.argsort(-r, axis=-1, kind="stable")[:, :k]
    keep = np.ones(shape, bool)
    np.put_along_axis(keep, idx, False, axis=-1)
    return keep


# --------------------------------------------------------------------------------------------
# floating-point path (torch fp32 on CPU)
# --------------------------------------------------------------------------------------------

def layer_norm(x, gamma):
    """transformer.py:24-31: bias-less LayerNorm (beta is a zero buffer), eps 1e-5."""
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return (x - mu) * torch.rsqrt(var + 1e-5) * gamma


def t5_bucket(relative_position: torch.Tensor, num_buckets=32, max_distance=128) -> torch.Tensor:
    """T5RelativePositionBias._relative_position_bucket (causal), transformer.py:86-104.  NB: it is fed i - j and negates
    it (n = j - i, clamped at 0), so every causally visible pair (j <= i) lands in bucket 0."""
    n = torch.max(-relative_position, torch.zeros_like(relative_position))
    max_exact = num_buckets // 2
    is_small = n < max_exact
    val_if_large = max_exact + (torch.log(n.float() / max_exact) / math.log(max_distance / max_exact) * (num_buckets - max_exact)).long()
    val_if_large = torch.min(val_if_large, torch.full_like(val_if_large, num_buckets - 1))
    return torch.where(is_small, n, val_if_large)


def rel_pos_table(sd, n: int, bias_type: str = "continuous", heads: int = 0, dtype=torch.float32) -> torch.Tensor:
    """RelativePositionBias.forward, transformer.py:55-67, restricted to the causal side: returns
    table[h, delta] for delta = i - j in [0, n).  (The reference evaluates the MLP on all 2n-1
    distances and gathers [h, i, j]; entries with j > i are overwritten by the causal mask.)
    't5': T5RelativePositionBias.forward, transformer.py:106-117 (bucket of i - j, see t5_bucket); 'none': zeros
    (transformer.py:372-373: no bias is added).  dtype: the precision the table is computed in (float64 for the
    kernel tests); the parameters are cast to it differentiably."""
    if bias_type == "none":
        return torch.zeros(heads, n, dtype=dtype)
    if bias_type == "t5":
        w = sd["transformer.rel_pos_bias.relative_attention_bias.weight"]
        bucket = t5_bucket(torch.arange(n, device=w.device))       # delta = i - j >= 0
        return w.to(dtype)[bucket].t().contiguous()
    p = lambda k: sd[f"transformer.rel_pos_bias.net.{k}"].to(dtype)
    x = torch.arange(n, dtype=dtype, device=p("0.0.weight").device)[:, None]
    for j in range(3):
        x = F.silu(x @ p(f"{j}.0.weight").t() + p(f"{j}.0.bias"))
    x = x @ p("3.weight").t() + p("3.bias")
    return x.t().contiguous()


def attention(cfg: Cfg, sd, p: str, x, table, key_mask):
    """Attention.forward (self-attention, causal), transformer.py:214-333."""
    B, N, _ = x.shape
    h, dh = cfg.heads, cfg.dim_head
    xn = layer_norm(x, sd[p + "norm.gamma"])                                                    # :250
    q = xn @ sd[p + "to_q.weight"].t()                                                          # :254
    # NB: kv_input is bound to the PRE-norm x at :228, before `x = self.norm(x)` at :250, so keys and
    # values are projected from the raw residual stream while queries see the normalised one.
    kv = x @ sd[p + "to_kv.weight"].t()                                                         # :228, :254
    k, v = kv[..., :dh], kv[..., dh:]
    q = q.view(B, N, h, dh).permute(0, 2, 1, 3)                                                 # :265
    q = q / q.norm(dim=-1, keepdim=True).clamp_min(1e-12) * sd[p + "q_scale"]                   # :269-271, utils.py:68-69
    k = k / k.norm(dim=-1, keepdim=True).clamp_min(1e-12) * sd[p + "k_scale"]
    sim = torch.einsum("bhid,bjd->bhij", q, k) * cfg.attn_scale                                 # :304
    i = torch.arange(N)
    delta = i[:, None] - i[None, :]
    bias = table[:, delta.clamp_min(0)]                                                         # :306-308 (j<=i side)
    sim = sim + bias[None]
    neg = -torch.finfo(sim.dtype).max
    if key_mask is not None:
        sim = sim.masked_fill(~key_mask[:, None, None, :], neg)                                 # :310-313
    sim = sim.masked_fill((delta < 0)[None, None], neg)                                         # :315-322
    attn = sim.softmax(-1)                                                                      # :324
    o = torch.einsum("bhij,bjd->bhid", attn, v).permute(0, 2, 1, 3).reshape(B, N, h * dh)       # :328-331
    return o @ sd[p + "to_out.0.weight"].t()                                                    # :333


def conv_feed_forward(cfg: Cfg, sd, p: str, x, drop_keep=None):
    """ConvFeedForward, transformer.py:140-150 (CausalDSConv 122-131, GEGLU 134-137), or the plain FeedForward
    (transformer.py:152-161: same chain without the depthwise conv, inner width 4 d) when cfg.use_conv_ff is False.
    drop_keep: optional [B, N, F] boolean keep-mask for the inner dropout (training)."""
    Fi = cfg.ff_inner
    k_g1, k_w1, k_conv, k_gin, k_w2 = cfg.ff_keys
    xn = layer_norm(x, sd[p + k_g1])
    y = xn @ sd[p + k_w1].t()                                                                   # :144 / :156
    if k_conv is not None:
        w = sd[p + k_conv][:, 0, :]                                                             # [2F, 3]
        up = F.pad(y, (0, 0, 2, 0))                                                             # left-pad time by 2 (:129)
        y = up[:, 0:-2] * w[:, 0] + up[:, 1:-1] * w[:, 1] + up[:, 2:] * w[:, 2]                 # :130
    a, g = y[..., :Fi], y[..., Fi:]                                                             # :136
    hmid = F.gelu(g) * a                                                                        # :137 (exact erf)
    hn = layer_norm(hmid, sd[p + k_gin])                                                        # :147 / :158
    if drop_keep is not None:
        hn = hn * drop_keep / (1.0 - cfg.ff_dropout)                                            # :148 / :159
    return hn @ sd[p + k_w2].t()                                                                # :149 / :160


def transformer_trunk(cfg: Cfg, sd, x, key_mask, drop_keeps=None):
    """Transformer.forward, transformer.py:385-424 (grad_shrink is the identity in forward)."""
    N = x.shape[1]
    a = cfg.grad_shrink_alpha
    x = x * a + x.detach() * (1 - a)                                                            # :400, utils.py:60-61
    table = rel_pos_table(sd, N, cfg.rel_pos_bias_type, cfg.heads)                              # :402-405
    for l in range(cfg.depth):
        p = f"transformer.layers.{l}."
        x = attention(cfg, sd, p + "0.", x, table, key_mask) + x                                # :415
        x = conv_feed_forward(cfg, sd, p + "2.", x, None if drop_keeps is None else drop_keeps[l]) + x  # :422
    return layer_norm(x, sd["transformer.norm.gamma"])                                          # :424


def embed(cfg: Cfg, sd, ids: Sequence[np.ndarray]) -> torch.Tensor:
    """open_musiclm.py:123-145: [start_s, embeddings_s[rows]] per sequence, concatenated."""
    parts = []
    B = ids[0].shape[0]
    for s, (rows, pad) in enumerate(embedding_rows(cfg, ids)):
        e = sd[f"embeddings.{s}.weight"][torch.from_numpy(rows)]
        e = e.masked_fill(torch.from_numpy(pad)[..., None], 0.0)                                # utils.py:137-138
        if cfg.abs_pos:                                                                         # open_musiclm.py:134-136
            e = e + sd[f"absolute_position_embeddings.{s}.weight"][:e.shape[1]][None]
        parts.append(sd[f"start_tokens.{s}"][None, None, :].expand(B, 1, -1))
        parts.append(e)
    return torch.cat(parts, 1)


def logits_from_hidden(cfg: Cfg, sd, hidden, seq_lens: Sequence[int], only_final=False):
    """open_musiclm.py:149-190: split at sequence boundaries, drop the next-start position of every
    sequence but the last, per-quantizer heads chosen by position mod q (remainder: heads 0..r-1)."""
    out, pos = [], 0
    S = len(cfg.seqs)
    for s, (info, n_tok) in enumerate(zip(cfg.seqs, seq_lens)):
        span = n_tok + 1                                  # start token + tokens
        hs = hidden[:, pos:pos + span]
        pos += span
        if s < S - 1:
            hs = hs[:, :-1]                                                                     # :156
        if only_final and s < S - 1:
            out.append(None)
            continue
        W = sd[f"logit_weights.{s}"]                      # [q, C+1, d]
        n, q = hs.shape[1], info.num_quantizers
        lg = hs.new_empty(hs.shape[0], n, W.shape[1])
        for qi in range(min(q, n)):                       # position p uses head p mod q, remainder included (:166-182)
            lg[:, qi::q] = hs[:, qi::q] @ W[qi].t()
        out.append(lg)
    return out


def forward_logits(cfg: Cfg, sd, ids: Sequence[np.ndarray], key_mask: Optional[np.ndarray], only_final=False, drop_keeps=None):
    """TokenConditionedTransformer.forward, open_musiclm.py:100-190."""
    x = embed(cfg, sd, ids)
    km = None if key_mask is None else torch.from_numpy(key_mask)
    hidden = transformer_trunk(cfg, sd, x, km, drop_keeps)
    return logits_from_hidden(cfg, sd, hidden, [t.shape[1] for t in ids], only_final)


def wrapper_loss(cfg: Cfg, all_logits, labels):
    """open_musiclm.py:389-410: token-count-weighted CE.  num_logits stays 0 for a sequence whose
    weight is 0 (:395,398-399), so the denominator counts only the weighted sequences."""
    weights = cfg.ce_weights if cfg.ce_weights is not None else [1.0] * len(cfg.seqs)
    total, running = 0, 0.0
    for lg, lb, w in zip(all_logits, labels, weights):
        n = 0
        loss = 0.0
        if w > 0 and lg is not None:
            n = int(lb.size)                                                                    # :399
            loss = F.cross_entropy(lg.reshape(-1, lg.shape[-1]), torch.from_numpy(lb).reshape(-1))  # :401
        total += n
        running = running + loss * n * w
    return running / total


def loss_and_logits(cfg: Cfg, sd, all_token_ids: Sequence[np.ndarray], forget_mask=None, drop_keeps=None):
    """TokenConditionedTransformerWrapper.forward(return_loss=True), open_musiclm.py:328-410."""
    ids, mask, labels = prepare_ids(cfg, all_token_ids, True, forget_mask)
    logits = forward_logits(cfg, sd, ids, mask, drop_keeps=drop_keeps)
    return wrapper_loss(cfg, logits, labels), logits, labels, ids, mask


# --------------------------------------------------------------------------------------------
# optimiser step (trainer.py:443-449, optimizer.py:10-40) on a dict of params / grads
# --------------------------------------------------------------------------------------------

def clip_and_adamw(params: Dict[str, torch.Tensor], grads: Dict[str, torch.Tensor], state: Dict[str, dict], *,
                   step: int, lr=3e-4, wd=1e-2, betas=(0.9, 0.99), eps=1e-8, max_grad_norm=0.5,
                   warmup_iters=0, start_factor=1e-7) -> float:
    """One SingleStageTrainer optimiser update: clip_grad_norm_(max_grad_norm) (trainer.py:443-444),
    AdamW with weight decay only on ndim>=2 params (optimizer.py:3-34), LinearLR warm-up factor for
    this step (optimizer.py:36-40; `step` = number of scheduler.step() calls so far).  In place.
    Returns the pre-clip global grad norm."""
    names = [k for k in params if k in grads and grads[k] is not None]
    total = math.sqrt(sum(float((grads[k].double() ** 2).sum()) for k in names))
    coef = min(1.0, max_grad_norm / (total + 1e-6))
    if warmup_iters > 0:
        fac = start_factor + (1.0 - start_factor) * min(step, warmup_iters) / warmup_iters
    else:
        fac = 1.0
    cur_lr = lr * fac
    b1, b2 = betas
    for k in names:
        g = grads[k] * coef
        st = state.setdefault(k, {"t": 0, "m": torch.zeros_like(params[k]), "v": torch.zeros_like(params[k])})
        st["t"] += 1
        t = st["t"]
        decay = wd if params[k].ndim >= 2 else 0.0
        params[k].mul_(1.0 - cur_lr * decay)
        st["m"].mul_(b1).add_(g, alpha=1 - b1)
        st["v"].mul_(b2).addcmul_(g, g, value=1 - b2)
        denom = (st["v"].sqrt() / math.sqrt(1 - b2 ** t)).add_(eps)
        params[k].addcdiv_(st["m"], denom, value=-cur_lr / (1 - b1 ** t))
    return total


# --------------------------------------------------------------------------------------------
# autoregressive generation (TokenConditionedTransformerWrapper.generate, open_musiclm.py:253-326)
# --------------------------------------------------------------------------------------------

def top_k_filter(logits: torch.Tensor, thres: float) -> torch.Tensor:
    """utils.py:78-84: keep the k = max(int((1 - thres) * C), 1) largest logits, -inf elsewhere."""
    k = max(int((1 - thres) * logits.shape[-1]), 1)
    val, ind = torch.topk(logits, k)
    out = torch.full_like(logits, float("-inf"))
    out.scatter_(1, ind, val)
    return out


def gumbel_argmax(logits: torch.Tensor, uniform: torch.Tensor, temperature: float) -> torch.Tensor:
    """utils.py:71-76 given the uniform(0,1) draw: argmax(logits / T - log(-log(u + 1e-20) + 1e-20))."""
    noise = -torch.log(-torch.log(uniform + 1e-20) + 1e-20)
    return (logits / temperature + noise).argmax(dim=-1)


def generate(cfg: Cfg, sd, conditioning_token_ids: Sequence[np.ndarray], uniforms, pred_token_ids: Optional[np.ndarray] = None,
             max_time_steps=8, filter_thres=0.9, temperature=1.0, include_eos_in_output=False, allow_eos_in_output=False,
             return_trace=False):
    """TokenConditionedTransformerWrapper.generate, open_musiclm.py:253-326, for unique_consecutive=False sequences:
    eos appended to every conditioning sequence (:288-290; ids are NOT zeroed and there is NO key mask at inference),
    the full prefix is re-run for every new token (:303-307), eos is forbidden except at the last quantizer of a time
    step when allow_eos_in_output (:311-313), top-k (utils.py:78-84) then Gumbel-argmax (utils.py:71-76), finally
    everything after an eos is set to -1 (:321-322, utils.py:86-93) and the flat ids are folded to [b, n, q] (:323-324).
    `uniforms(step, shape)` supplies the uniform(0,1) draw of gumbel_noise for each sampled token, in order.
    return_trace: also return per-step (logits of the last position, gap between the best and second-best noisy score)."""
    S = len(cfg.seqs)
    assert len(conditioning_token_ids) == S - 1
    B = conditioning_token_ids[0].shape[0]
    cond = [np.asarray(t).reshape(B, -1).astype(np.int64) for t in conditioning_token_ids]
    cond = [np.concatenate([t, np.full((B, 1), s.codebook_size, np.int64)], 1) for t, s in zip(cond, cfg.seqs)]   # :288-290
    info = cfg.seqs[-1]
    eos = info.codebook_size
    if pred_token_ids is not None:
        init_step = pred_token_ids.shape[1]                                                                        # :276
        pred = np.asarray(pred_token_ids).reshape(B, -1).astype(np.int64)
    else:
        init_step = 0
        pred = np.zeros((B, 0), np.int64)
    trace = []
    step = 0
    with torch.no_grad():
        for _t in range(init_step, max_time_steps):
            for ind in range(info.num_quantizers):
                last = ind == info.num_quantizers - 1
                lg = forward_logits(cfg, sd, cond + [pred], None, only_final=True)[-1][:, -1].clone()             # :303-309
                if not allow_eos_in_output or not last:
                    lg[:, -1] = float("-inf")                                                                      # :311-313
                filt = top_k_filter(lg, filter_thres)
                u = uniforms(step, tuple(filt.shape))
                noisy = filt / temperature + (-torch.log(-torch.log(u + 1e-20) + 1e-20))
                top2 = torch.topk(noisy, 2, dim=-1).values
                sampled = noisy.argmax(dim=-1)
                trace.append((lg, (top2[:, 0] - top2[:, 1]).clone()))
                pred = np.concatenate([pred, sampled.numpy()[:, None]], 1)                                          # :318-319
                step += 1
    out = torch.from_numpy(pred)
    eos_mask = (out == eos).float()
    if include_eos_in_output:
        eos_mask = F.pad(eos_mask, (1, -1))                                                                        # utils.py:89-90
    out = out.masked_fill(eos_mask.cumsum(-1) > 0, -1)
    out = out.view(B, -1, info.num_quantizers)
    return (out, trace) if return_trace else out
