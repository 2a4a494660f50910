"""CPU: the C-ABI library builds, loads and exports every symbol include/parseq_b200.h declares; the
host-side mirror of the reference interface (factory, hub entry points, tokenizer) behaves like the reference's;
and the product path fails loudly without a GPU (no CPU fallback)."""
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SURFACE = torch.load(os.path.join(ROOT, "tests", "golden", "reference", "surface.pt"), weights_only=False)


def test_library_exports_every_declared_symbol(lib):
    hdr = open(os.path.join(ROOT, "include", "parseq_b200.h")).read()
    declared = set(re.findall(r"\b(parseq_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"parseq_status"}
    assert len(declared) >= 15
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    from parseq_b200.engine import EXPORTS
    assert set(EXPORTS) == declared
    assert b"sm_100a" in lib.parseq_version()


def test_launch_options_documented_in_the_header_are_accepted(lib):
    """Every launch option the header names is accepted on the NULL handle (process defaults; no CUDA call involved), range
    errors and unknown names are reported through the status code."""
    from parseq_b200.engine import check
    names = ["block_n", "attn_impl", "pdl", "tma_epilogue", "gemm_stages", "cta_group", "ln_cta_group", "mlp_cta_group", "pair_pdl",
             "ln_split"]
    hdr = open(os.path.join(ROOT, "include", "parseq_b200.h")).read()
    for n in names:
        assert f'"{n}"' in hdr or n in hdr, n
        default = 1 if n in ("attn_impl", "pdl", "tma_epilogue") else 0
        check(lib, lib.parseq_set_option(None, n.encode(), default))
    for n, bad in (("cta_group", 3), ("ln_cta_group", -1), ("mlp_cta_group", 5), ("ln_split", 3), ("block_n", 100)):
        assert lib.parseq_set_option(None, n.encode(), bad) != 0
        assert lib.parseq_last_error()
        check(lib, lib.parseq_set_option(None, n.encode(), 0))
    assert lib.parseq_set_option(None, b"fuse_mlp", 1) != 0          # per-handle options need a handle
    assert lib.parseq_set_option(None, b"no_such_option", 1) != 0


def test_sass_is_blackwell_native():
    """The GEMM kernel must contain tcgen05 / TMA / TMEM instructions (UTCHMMA, UTMALDG, LDTM)."""
    import shutil
    import subprocess
    from parseq_b200.build import LIB_PATH, build
    build()
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([cuobjdump, "-sass", LIB_PATH], capture_output=True, text=True).stdout
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):
        assert mnemonic in sass, mnemonic
    assert "sm_100a" in sass or "sm_100" in sass
    # the fused residual-GEMM + LayerNorm kernel: UMMA + TMA load AND store + TMEM load AND store (the updated row is
    # parked in TMEM between its two epilogue passes)
    fn = [b for b in sass.split("Function : ")[1:] if "gemm_ln_fused_kernel" in b.split("\n", 1)[0]]
    assert len(fn) == 4                       # D in {192, 384} x {single CTA, CTA pair}
    for body in fn:
        for mnemonic in ("UTCHMMA", "UTMALDG", "UTMASTG", "LDTM", "STTM"):
            assert mnemonic in body, mnemonic
    # its column-split CTA-pair version: the same inside a cluster (hardware cluster barrier; the statistics go to the peer by distributed shared memory)
    fn = [b for b in sass.split("Function : ")[1:] if "gemm_ln_split_kernel" in b.split("\n", 1)[0]]
    assert len(fn) == 1
    for mnemonic in ("UTCHMMA", "UTMALDG", "UTMASTG", "LDTM", "STTM", "UCGABAR"):
        assert mnemonic in fn[0], mnemonic
    # the cluster-owned AR kernel: TMA loads into its ring, hardware cluster barriers, warp MMA (10 instantiations)
    fn = [b for b in sass.split("Function : ")[1:] if "dec_ar2_kernel" in b.split("\n", 1)[0]]
    assert len(fn) == 12                      # D in {192, 384} x MT in {1, 2} x cluster size {6, 8}, D = 768 x {6, 8}, head-split D in {192, 384}
    for body in fn:
        for mnemonic in ("UTMALDG", "UCGABAR", "HMMA", "LDSM"):
            assert mnemonic in body, mnemonic
    # tcgen05 attention for T = 128 and the two-key-block variant for any T <= 256
    fn = [b for b in sass.split("Function : ")[1:] if "enc_attention_tc" in b.split("\n", 1)[0]]
    assert len(fn) == 3
    for body in fn:
        for mnemonic in ("UTCHMMA", "UTMALDG", "UTMASTG", "LDTM"):
            assert mnemonic in body, mnemonic
    # the fc1 epilogue evaluates GELU on packed fp32 pairs
    fn = [b for b in sass.split("Function : ")[1:] if "gemm_bf16_tcgen05_kernel" in b.split("\n", 1)[0]]
    assert fn and all("FFMA2" in body for body in fn)


def test_no_cpu_fallback():
    from parseq_b200.factory import create_model
    m = create_model("parseq")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 3, 32, 128))
    if not torch.cuda.is_available():
        from parseq_b200.config import make_config
        from parseq_b200.engine import Engine, EngineError
        with pytest.raises(EngineError):
            Engine(make_config("parseq"), 0)


def test_factory_and_hub_entry_points():
    import hubconf
    from strhub.models.utils import create_model, parse_model_args, InvalidModelError
    from strhub.models.parseq.system import PARSeq
    m = create_model("parseq-tiny", decode_ar=False, refine_iters=3, name="x", _convert_="all")
    assert isinstance(m, PARSeq)
    assert m.hparams.embed_dim == 192 and m.hparams.refine_iters == 3 and m.model.refine_iters == 3
    assert not m.model.decode_ar and m.hparams.charset_test == "0123456789abcdefghijklmnopqrstuvwxyz"
    assert len(m.tokenizer) == 97 and (m.eos_id, m.bos_id, m.pad_id) == (0, 95, 96)
    assert hubconf.parseq_tiny().hparams.img_size == [32, 128]
    with pytest.raises(InvalidModelError):
        create_model("crnn")
    assert parse_model_args(["refine_iters:int=2", "decode_ar:bool=false", "lr:float=1e-3", "name:str=a"]) == {
        "refine_iters": 2, "decode_ar": False, "lr": 1e-3, "name": "a"}


def test_state_dict_keys_match_reference_layout():
    from parseq_b200.factory import create_model
    sd = create_model("parseq").model.state_dict()
    assert len(sd) == 175
    assert tuple(sd["encoder.patch_embed.proj.weight"].shape) == (384, 3, 4, 8)
    assert tuple(sd["decoder.layers.0.cross_attn.in_proj_weight"].shape) == (1152, 384)
    assert tuple(sd["pos_queries"].shape) == (1, 26, 384)
    assert tuple(sd["head.weight"].shape) == (95, 384)
    assert tuple(sd["text_embed.embedding.weight"].shape) == (97, 384)
    # the reference model's own state_dict (tests/golden/reference, oracle/make_golden.py): a strict load needs the same
    # names and shapes
    ref = REF_SURFACE["state_dict_shapes"]
    assert set(ref) == set(sd)
    assert all(tuple(sd[k].shape) == ref[k] for k in ref)


def test_tokenizer_matches_reference_semantics():
    from strhub.data.utils import Tokenizer, CharsetAdapter
    from parseq_b200.config import CHARSET_94
    tok = Tokenizer(CHARSET_94)
    enc = tok.encode(["ab", "hello!"])
    assert enc.shape == (2, 8) and enc[0, 0] == 95 and enc[0, 3] == 0 and enc[0, 4] == 96
    probs = torch.zeros(2, 5, 95)
    seq = [[11, 12, 0, 13, 14], [36 + 1, 1, 2, 3, 4]]
    for b in range(2):
        for i, t in enumerate(seq[b]):
            probs[b, i, t] = 0.9
    labels, ps = tok.decode(probs)
    assert labels == ["ab", "A0123"] and len(ps[0]) == 3 and len(ps[1]) == 5
    assert CharsetAdapter("0123456789abcdefghijklmnopqrstuvwxyz")("Ab-C9") == "abc9"
    # the reference Tokenizer on the same inputs (tests/golden/reference, oracle/make_golden.py)
    ref = REF_SURFACE
    assert ref["charset"] == CHARSET_94 and torch.equal(ref["decode_probs"], probs)
    assert ref["decode_labels"] == labels and len(ref["decode_token_probs"]) == len(ps)
    assert all(torch.equal(a, b) for a, b in zip(ref["decode_token_probs"], ps))
    assert ref["encode_texts"] == ["ab", "hello!"] and torch.equal(ref["encode_ids"], enc)


def test_edit_distance():
    from parseq_b200.system import edit_distance
    assert edit_distance("kitten", "sitting") == 3 and edit_distance("", "abc") == 3 and edit_distance("a", "a") == 0
