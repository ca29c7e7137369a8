"""ORACLE — test infrastructure only.  Generates tests/golden/reference_checks.pt from the REAL reference.

Run where the reference tree is importable (oracle/ref_harness.py):   python oracle/make_golden_checks.py
The fixture holds what the reference computed for four comparisons, so that the tests run without it:
  init     per parameter, the SHA-256 of the reference's initial weights under torch.manual_seed(0), for every stage
           and three configuration variants (tests/test_boundary_cpu.py)
  crops    the token crops of the reference's PreprocessedDataset.__getitem__ over a synthetic sqlite database
           (tests/test_data_cpu.py)
  mask     the reference's forgetful mask (utils.generate_mask_with_prob) under a fixed seed (tests/test_oracle_cpu.py)
  live     a mid-size model per stage: the digest of the reference's weights, the input tokens, the loss and a fixed,
           seeded sample of every logits tensor (tests/test_oracle_cpu.py)
"""
import hashlib
import importlib
import os
import random
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.make_golden import GOLD  # noqa: E402

PATH = os.path.join(GOLD, "reference_checks.pt")

INIT_BASE = dict(dim=128, depth=2, heads=2, attn_dropout=0.0, ff_dropout=0.1)
INIT_VARIANTS = [dict(), dict(use_conv_ff=False, relative_position_bias_type="t5"),
                 dict(relative_position_bias_type="none", use_absolute_position_embeddings=True)]
STAGES = ["semantic", "coarse", "fine"]

LIVE_COMMON = dict(attn_dropout=0.0, ff_dropout=0.1, grad_shrink_alpha=0.1, non_causal_prefix_size=0,
                   relative_position_bias_type="continuous", use_memory_efficient_attention=False)
LIVE = {  # stage: (model kwargs, token shapes, ce weights)
    "semantic": (dict(dim=192, depth=2, heads=3), [(2, 12), (2, 40)], [0.0, 1.0]),
    "coarse": (dict(dim=192, depth=2, heads=3, num_coarse_quantizers=3), [(2, 12), (2, 20), (2, 9, 3)], [0.0, 0.0, 1.0]),
    "fine": (dict(dim=192, depth=2, heads=3, num_coarse_quantizers=3, num_fine_quantizers=5), [(2, 12), (2, 5, 3), (2, 5, 5)],
             [0.0, 0.0, 1.0]),
}
LIVE_SAMPLE = 1024      # logits entries kept per tensor


def digest(t: torch.Tensor) -> str:
    return hashlib.sha256(t.detach().contiguous().cpu().numpy().tobytes()).hexdigest()


def state_digests(sd):
    return [(k, tuple(v.shape), str(v.dtype), digest(v)) for k, v in sd.items()]


def main():
    from oracle import ref_harness
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_data_cpu import synth_items
    from open_musiclm_b200 import data as D
    ref = ref_harness.import_reference()
    utils = sys.modules["open_musiclm.utils"]
    create = {s: getattr(ref, f"create_{s}_transformer") for s in STAGES}

    init = []
    for extra in INIT_VARIANTS:
        kw = dict(INIT_BASE, **extra)
        per_stage = {}
        for s in STAGES:
            torch.manual_seed(0)
            per_stage[s] = state_digests(create[s](**kw).state_dict())
        init.append({"kwargs": kw, "stages": per_stage})

    ref_data = importlib.import_module("open_musiclm.data")
    items = synth_items(5, seed=3)
    crops = {}
    with tempfile.TemporaryDirectory() as tmp:
        D.write_sqlite(tmp, items)
        for s in STAGES:
            ds = ref_data.PreprocessedDataset(tmp, s)
            per_item = []
            for idx in range(len(ds)):
                random.seed(100 + idx)
                per_item.append([t.to(torch.int16) for t in ds[idx]])
            crops[s] = per_item

    torch.manual_seed(11)
    mask = utils.generate_mask_with_prob((4, 50), 0.15, device="cpu")

    live = {}
    for s, (kw, shapes, cew) in LIVE.items():
        torch.manual_seed(5)
        model = create[s](**kw, **LIVE_COMMON)
        wrapper = ref.TokenConditionedTransformerWrapper(transformer=model, unique_consecutive=False,
                                                         cross_entropy_loss_weights=cew).eval()
        g = torch.Generator().manual_seed(99)
        toks = [torch.randint(0, 1024, sh, generator=g) for sh in shapes]
        with torch.no_grad():
            loss, logits, _ = wrapper(all_token_ids=[t.clone() for t in toks], return_loss=True)
        gs = torch.Generator().manual_seed(2024)
        samples = []
        for l in logits:
            l = l.permute(0, 2, 1).contiguous()                                    # [b, n, c], as the restatement returns it
            idx = torch.randperm(l.numel(), generator=gs)[:LIVE_SAMPLE].sort().values
            samples.append({"shape": tuple(l.shape), "index": idx.to(torch.int32), "value": l.reshape(-1)[idx].clone()})
        live[s] = {"kwargs": dict(kw, **LIVE_COMMON), "ce_weights": cew, "state": state_digests(model.state_dict()),
                   "tokens": toks, "loss": loss.detach().double(), "logits": samples}

    torch.save({"init": init, "crops": crops, "mask": mask, "live": live}, PATH)
    print(PATH, os.path.getsize(PATH) // 1024, "KiB")


if __name__ == "__main__":
    main()
