"""CPU checks of the drop-in boundary: C ABI exports, state_dict contract, init parity, loud failure without a GPU."""
import ctypes
import glob
import os

import pytest
import torch

import open_musiclm_b200 as O
from open_musiclm_b200 import lib
from oracle.make_golden_checks import digest

GOLD = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "tiny_*.pt")))
CHECKS = os.path.join(os.path.dirname(__file__), "golden", "reference_checks.pt")


def build_from_fixture(fx):
    fn = {"semantic": O.create_semantic_transformer, "coarse": O.create_coarse_transformer, "fine": O.create_fine_transformer}[fx["stage"]]
    return fn(**fx["kwargs"])


def test_abi_library_exports_every_declared_symbol():
    l = lib.load()
    syms = lib.header_symbols()
    assert len(syms) >= 25
    for s in syms:
        assert hasattr(l, s), f"{s} declared in include/omlm_b200.h but not exported"
    assert l.omlm_abi_version() == 2
    l.omlm_last_error.restype = ctypes.c_char_p
    assert isinstance(l.omlm_last_error(), bytes)


@pytest.mark.parametrize("path", GOLD, ids=[os.path.basename(p) for p in GOLD])
def test_state_dict_contract_matches_reference_fixture(path):
    fx = torch.load(path, weights_only=False)
    m = build_from_fixture(fx)
    sd = m.state_dict()
    assert list(sd.keys()) == list(fx["state_dict"].keys())
    for k, v in fx["state_dict"].items():
        assert sd[k].shape == v.shape and sd[k].dtype == v.dtype, k
    m.load_state_dict(fx["state_dict"], strict=True)
    names = [n for n, _ in m.named_parameters()]
    assert names == list(fx["grads"].keys())          # same parameters, same order as the reference
    assert m.eos_ids == [s.codebook_size for s in m.token_sequences]
    assert m.token_sequences[-1].num_quantizers >= 1 and not m.has_condition


def test_init_is_bit_identical_to_reference_under_same_seed():
    """Initial weights under torch.manual_seed(0) against the SHA-256 of the reference's, parameter by parameter
    (tests/golden/reference_checks.pt, oracle/make_golden_checks.py)."""
    init = torch.load(CHECKS, weights_only=False)["init"]
    assert len(init) == 3
    for case in init:
        kw = case["kwargs"]
        for stage, theirs in case["stages"].items():
            torch.manual_seed(0)
            a = getattr(O, f"create_{stage}_transformer")(**kw).state_dict()
            assert [k for k, *_ in theirs] == list(a.keys()), (kw, stage)
            for k, shape, dtype, sha in theirs:
                assert tuple(a[k].shape) == shape and str(a[k].dtype) == dtype, (kw, stage, k)
                assert digest(a[k]) == sha, (kw, stage, k)


def test_no_cpu_fallback():
    m = O.create_semantic_transformer(dim=64, depth=1, heads=1, clap_codebook_size=16, semantic_codebook_size=16, num_clap_quantizers=2)
    with pytest.raises(lib.OmlmError):
        m(all_token_ids=[torch.zeros(1, 2, dtype=torch.long), torch.zeros(1, 3, dtype=torch.long)])


def test_unsupported_configs_fail_loudly():
    for kw in [dict(non_causal_prefix_size=4), dict(attn_dropout=0.1), dict(use_memory_efficient_attention=True),
               dict(has_condition=True)]:
        with pytest.raises(NotImplementedError):
            O.create_semantic_transformer(dim=64, depth=1, heads=1, **kw)


def test_pack_job_struct_matches_header():
    """lib._PackJob (ctypes) mirrors `omlm_pack_job` of include/omlm_b200.h field for field: the job table is built on
    the host and read by omlm_pack_multi on the device."""
    import ctypes
    import re
    from open_musiclm_b200 import lib
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "omlm_b200.h")).read()
    body = re.search(r"typedef struct \{(.*?)\} omlm_pack_job;", hdr, re.S).group(1)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        for part in decl.split(","):
            names.append(re.sub(r"[\s\*]", " ", part).split()[-1])
    assert names == [f[0] for f in lib._PackJob._fields_]
    assert ctypes.sizeof(lib._PackJob) == 3 * 8 + 3 * 8 + 8 * 4
    assert lib._PackJob.unit_start.offset == 40 and lib._PackJob.rows_valid.offset == 48


def test_decode_layer_struct_matches_header():
    """lib._DecodeLayer (ctypes) mirrors `omlm_decode_layer` of include/omlm_b200.h field for field: the per-layer pointer table of
    the fused decode step is built on the host and read by omlm_decode_step on the device."""
    import ctypes
    import re
    from open_musiclm_b200 import lib
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "omlm_b200.h")).read()
    end = hdr.index("} omlm_decode_layer;")
    body = hdr[hdr.rindex("typedef struct {", 0, end) + len("typedef struct {"):end]
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        for part in decl.split(","):
            names.append(re.sub(r"[\s\*]", " ", part).split()[-1])
    assert names == [f[0] for f in lib._DecodeLayer._fields_]
    assert ctypes.sizeof(lib._DecodeLayer) == 13 * 8
