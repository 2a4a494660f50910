"""Generates tests/golden/*.pt by running the UNMODIFIED reference modules
(/root/reference/strhub/models/parseq/model.py under oracle/timm_shim.py) on seeded synthetic
weights and crops.  Run in the build container (the GPU box has no /root/reference):

    python -m oracle.make_golden [vitstr | sharp | reference | filtered ...]

TEST INFRASTRUCTURE ONLY.  Weights are not stored: they are regenerated from (experiment, seed) by
parseq_b200.weights.init_state_dict and verified through `sd_digest`.
"""
from __future__ import annotations

import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from parseq_b200.config import make_config                      # noqa: E402
from parseq_b200.weights import init_state_dict, synth_images, state_dict_digest  # noqa: E402
from oracle import reference_loader as RL                        # noqa: E402
from oracle.parseq_oracle import ParseqOracle                    # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")

# (case name, experiment, weight seed, eos_bias, batch, image seed, decode_ar, refine_iters, max_length)
CASES = [
    ("s_ar1_b2",        "parseq",      0, 0.0, 2, 0, True,  1, None),
    ("s_ar1_b1",        "parseq",      0, 0.0, 1, 7, True,  1, None),
    ("s_ar0_b2",        "parseq",      0, 0.0, 2, 1, True,  0, None),
    ("s_nar0_b2",       "parseq",      0, 0.0, 2, 2, False, 0, None),
    ("s_nar3_b2",       "parseq",      0, 0.0, 2, 3, False, 3, None),
    ("s_ar3_b2",        "parseq",      0, 0.0, 2, 4, True,  3, None),
    ("s_ar1_len5_b2",   "parseq",      0, 0.0, 2, 5, True,  1, 5),
    ("s_ar0_len1_b2",   "parseq",      0, 0.0, 2, 5, True,  0, 1),
    ("s_eos_ar1_b4",    "parseq",      1, 0.5, 4, 6, True,  1, None),
    ("s_eos_ar0_b4",    "parseq",      1, 0.7, 4, 6, True,  0, None),
    ("s_eos_nar2_b4",   "parseq",      1, 0.5, 4, 8, False, 2, None),
    ("ti_nar0_b1",      "parseq-tiny", 2, 0.0, 1, 9, False, 0, None),
    ("ti_ar1_b3",       "parseq-tiny", 2, 0.0, 3, 10, True, 1, None),
    # other geometries: T = 196 tokens (224x224 / 16x16) and the BASELINE ViT-B-width stress config (48x160, T = 240, D = 768)
    ("p16_ar1_b2",      "parseq-patch16-224", 3, 0.0, 2, 11, True, 1, None),
    ("p16_nar1_b1",     "parseq-patch16-224", 3, 0.0, 1, 12, False, 1, None),
    ("b48_ar1_b2",      "parseq-base-48x160", 4, 0.0, 2, 13, True, 1, None),
]


# "sharp" cases (parseq_b200.weights._sharpen): q / k projections scaled 4x -> pre-softmax scores 16x -> peaked attention
# rows, so that a wrong / missing q, mask or scale shows up well above the bf16 tolerance.  One per embed width and
# decode mode.  Appended to CASES with a 10th field.
SHARP_CASES = [
    ("s_sharp_ar1_b2",   "parseq",             5, 0.0, 2, 20, True,  1, None, 4.0),
    ("s_sharp_nar2_b2",  "parseq",             5, 0.0, 2, 21, False, 2, None, 4.0),
    ("s_sharp_eos_ar1_b3", "parseq",           6, 0.6, 3, 22, True,  1, None, 4.0),
    ("ti_sharp_ar1_b3",  "parseq-tiny",        7, 0.0, 3, 23, True,  1, None, 4.0),
    ("ti_sharp_nar1_b2", "parseq-tiny",        7, 0.0, 2, 24, False, 1, None, 4.0),
    ("b48_sharp_ar1_b2", "parseq-base-48x160", 8, 0.0, 2, 25, True,  1, None, 4.0),
    ("p16_sharp_ar1_b2", "parseq-patch16-224", 9, 0.0, 2, 26, True,  1, None, 4.0),
]


def make_sd(experiment, seed, eos_bias, sharp=0.0):
    cfg = make_config(experiment)
    sd = init_state_dict(cfg, seed, sharp=sharp)
    if eos_bias:
        sd["head.bias"] = sd["head.bias"].clone()
        sd["head.bias"][0] += eos_bias
    return cfg, sd


def main(cases=None):
    assert RL.available(), "reference tree not present"
    os.makedirs(OUT, exist_ok=True)
    cache = {}
    for case in (cases if cases is not None else CASES + SHARP_CASES):
        name, exp, wseed, eos_bias, B, iseed, ar, ri, ml = case[:9]
        sharp = case[9] if len(case) > 9 else 0.0
        key = (exp, wseed, eos_bias, sharp)
        if key not in cache:
            cfg, sd = make_sd(exp, wseed, eos_bias, sharp)
            ref, tok = RL.build_reference_model(cfg, sd)
            cache[key] = (cfg, sd, ref, tok, ParseqOracle(cfg, sd, "fp64"))
        cfg, sd, ref, tok, o64 = cache[key]
        x = synth_images(cfg, B, iseed)
        ref.decode_ar, ref.refine_iters = ar, ri
        with torch.inference_mode():
            logits = ref(tok, x, ml).clone()
            memory = ref.encode(x).clone()
        o = o64.forward(x, ml, ar, ri)
        assert o.logits.shape == logits.shape, (name, o.logits.shape, logits.shape)
        err = (o.logits.float() - logits).abs().max().item()
        # pins the oracle (and its id trajectory) to the reference; the sharp cases amplify the reference's own fp32
        # round-off (fp64 oracle vs fp32 reference: 1.7e-5 at D = 768)
        assert err < (5e-5 if sharp else 1e-5), (name, err)
        bf16_err = None
        if sharp:
            # yardstick for the sharp cases: how far the rounding-point model of the engine (same graph, tensors rounded
            # to bf16 where the engine stores bf16 operands, fp32 accumulation) lands from the fp32 reference along the
            # same id trajectory.  Sharper attention amplifies operand rounding (D = 768: ~5x the plain cases), so the
            # GPU test bounds the engine by this measured figure instead of a constant.
            ob = ParseqOracle(cfg, sd, "bf16").forward(x, ml, ar, ri, forced_ids=o.ar_ids, forced_refine=o.refine_ctx)
            d = (ob.logits.float() - logits).abs()
            bf16_err = (float(d.max()), float(d.mean()))
        blob = dict(
            name=name, experiment=exp, weight_seed=wseed, eos_bias=eos_bias, sharp=sharp, batch=B, image_seed=iseed,
            bf16_model_err=bf16_err,
            decode_ar=ar, refine_iters=ri, max_length=ml, sd_digest=state_dict_digest(sd),
            logits=logits.contiguous(), memory0=memory[0].contiguous(),
            min_margin_fp64=o.min_margin.float(), steps=o.steps,
            # id trajectory of the reference run (for teacher-forced logit comparisons)
            ar_ids=None if o.ar_ids is None else o.ar_ids.int(),
            refine_ctx=[c.int() for c in o.refine_ctx],
            source="reference strhub.models.parseq.model.PARSeq @ /root/reference (timm shim), torch %s CPU fp32"
                   % torch.__version__,
        )
        torch.save(blob, os.path.join(OUT, name + ".pt"))
        print(f"{name:18s} logits {tuple(logits.shape)} S={o.steps} |ref-fp64 oracle|={err:.2e} "
              f"min margin {o.min_margin.min().item():.2e} bf16-model err {bf16_err}")


def make_filtered(name, exp, wseed, ar, ri, ml, n_blocks, block, tau, first_block=0):
    """Margin-filtered free-running set (SURVEY.md 7.2-1d): candidates whose smallest top1-top2 margin over
    every argmax decision of the fp32 reference run exceeds `tau`; on these, decoded ids must be bit-identical
    between the bf16 engine and the fp32 reference."""
    cfg, sd = make_sd(exp, wseed, 0.0)
    ref, tok = RL.build_reference_model(cfg, sd)
    ref.decode_ar, ref.refine_iters = ar, ri
    o32 = ParseqOracle(cfg, sd, "fp32")
    picks, ids, logits, margins, n_cand = [], [], [], [], 0
    for blk in range(first_block, first_block + n_blocks):
        seed = 90_000 + blk
        x = synth_images(cfg, block, seed)
        o = o32.forward(x, ml, ar, ri)
        n_cand += block
        keep = torch.nonzero(o.min_margin > tau).flatten().tolist()
        if keep:
            with torch.inference_mode():
                lr = ref(tok, x[keep], ml)          # the reference itself on the accepted images
            assert (lr - o.logits[keep]).abs().max().item() < 1e-5
            for j, k in enumerate(keep):
                picks.append((seed, k)); ids.append(lr[j].argmax(-1).int()); logits.append(lr[j].clone())
                margins.append(float(o.min_margin[k]))
        print(f"{name}: block {blk + 1}/{first_block + n_blocks} accepted so far {len(picks)}/{n_cand}", flush=True)
    blob = dict(name=name, experiment=exp, weight_seed=wseed, decode_ar=ar, refine_iters=ri, max_length=ml,
                block=block, tau=tau, candidates=n_cand, acceptance_rate=len(picks) / max(1, n_cand), picks=picks, ids=torch.stack(ids),
                logits=torch.stack(logits), margins=torch.tensor(margins), sd_digest=state_dict_digest(sd))
    torch.save(blob, os.path.join(OUT, name + ".pt"))


# (case name, config overrides, weight seed, batch, image seed, max_length)
VITSTR_CASES = [
    ("vitstr_s_b3",      dict(), 20, 3, 30, None),
    ("vitstr_s_len5_b2", dict(), 20, 2, 31, 5),
    ("vitstr_s_len0_b1", dict(), 20, 1, 32, 0),
    # configs/model/vitstr.yaml geometry (224x224 / 16x16: 196 patches + class token)
    ("vitstr_p16_b1",    dict(img_size=(224, 224), patch_size=(16, 16)), 21, 1, 33, None),
]


def make_vitstr():
    """Golden outputs of the reference's own `strhub.models.vitstr.model.ViTSTR` (under the timm shim) with the call and
    slice of vitstr/system.py:65-71."""
    from oracle.vitstr_oracle import VitstrOracle
    os.makedirs(OUT, exist_ok=True)
    for name, over, wseed, B, iseed, ml in VITSTR_CASES:
        cfg = make_config("vitstr", **over)
        sd = init_state_dict(cfg, wseed)
        ref = RL.build_reference_vitstr(cfg, sd)
        x = synth_images(cfg, B, iseed)
        m = cfg.max_label_length if ml is None else min(ml, cfg.max_label_length)
        with torch.inference_mode():
            logits = ref(x, m + 2)[:, 1:].clone()               # vitstr/system.py:67-70
            feats = ref.forward_features(x).clone()
        o = VitstrOracle(cfg, sd, "fp64")
        err = (o.system_forward(x, ml).float() - logits).abs().max().item()
        assert err < 1e-5, (name, err)
        blob = dict(name=name, experiment="vitstr", overrides=over, weight_seed=wseed, batch=B, image_seed=iseed,
                    max_length=ml, sd_digest=state_dict_digest(sd), logits=logits.contiguous(),
                    features0=feats[0].contiguous(),
                    source="reference strhub.models.vitstr.model.ViTSTR @ /root/reference (timm shim), torch %s CPU fp32"
                           % torch.__version__)
        torch.save(blob, os.path.join(OUT, name + ".pt"))
        print(f"{name:18s} logits {tuple(logits.shape)} |ref-fp64 oracle|={err:.2e}")


def make_reference_surface():
    """tests/golden/reference/: what the CPU tests compare against that is not a forward case of CASES — the reference
    PARSeq-Ti on one (weights, crops) pair under three decode schedules, the reference state_dict layout, and the
    reference Tokenizer on fixed inputs."""
    from parseq_b200.config import CHARSET_94
    out = os.path.join(OUT, "reference")
    os.makedirs(out, exist_ok=True)
    cfg, sd = make_sd("parseq-tiny", 11, 0.0)
    ref, tok = RL.build_reference_model(cfg, sd)
    x = synth_images(cfg, 2, 12)
    runs = []
    for ar, ri, ml in [(True, 1, None), (False, 0, None), (True, 2, 4)]:
        ref.decode_ar, ref.refine_iters = ar, ri
        with torch.inference_mode():
            runs.append(dict(decode_ar=ar, refine_iters=ri, max_length=ml, logits=ref(tok, x, ml).clone()))
    torch.save(dict(experiment="parseq-tiny", weight_seed=11, batch=2, image_seed=12, sd_digest=state_dict_digest(sd), runs=runs,
                    source="reference strhub.models.parseq.model.PARSeq (timm shim), torch %s CPU fp32" % torch.__version__),
               os.path.join(out, "tiny_w11_x12.pt"))

    cfg, sd = make_sd("parseq", 0, 0.0)
    ref, _ = RL.build_reference_model(cfg, sd)          # strict load
    shapes = {k: tuple(v.shape) for k, v in ref.state_dict().items()}
    _, RefTok = RL.load_reference_classes()
    rt = RefTok(CHARSET_94)
    # probabilities with a clear argmax per position: ids 11 12 | EOS 13 14 and 37 1 2 3 4 (no EOS)
    probs = torch.zeros(2, 5, 95)
    for b, seq in enumerate([[11, 12, 0, 13, 14], [36 + 1, 1, 2, 3, 4]]):
        for i, t in enumerate(seq):
            probs[b, i, t] = 0.9
    labels, ps = rt.decode(probs)
    texts = ["ab", "hello!"]
    torch.save(dict(state_dict_shapes=shapes, charset=CHARSET_94, decode_probs=probs, decode_labels=labels,
                    decode_token_probs=[p.clone() for p in ps], encode_texts=texts, encode_ids=rt.encode(texts),
                    source="reference strhub.models.parseq.model.PARSeq / strhub.data.utils.Tokenizer, torch %s"
                           % torch.__version__),
               os.path.join(out, "surface.pt"))
    print("reference surface:", len(shapes), "state_dict entries,", len(runs), "PARSeq-Ti runs")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "vitstr":
        make_vitstr()
    elif len(sys.argv) > 1 and sys.argv[1] == "reference":
        make_reference_surface()
    elif len(sys.argv) > 1 and sys.argv[1] == "sharp":
        main(SHARP_CASES)
    elif len(sys.argv) > 1 and sys.argv[1] == "filtered_ti":
        make_filtered("filtered_ti_ar1_len5", "parseq-tiny", 2, True, 1, 5, 4, 256, 0.012)
    elif len(sys.argv) > 1 and sys.argv[1] == "filtered_more":
        # extra candidate blocks [first, first + n) for the full-length set, written to <name>_part.pt; merge with
        # `python -m oracle.make_golden filtered_merge`
        first, n = int(sys.argv[2]), int(sys.argv[3])
        make_filtered("filtered_s_ar1_part", "parseq", 0, True, 1, None, n, 256, 0.02, first_block=first)
    elif len(sys.argv) > 1 and sys.argv[1] == "filtered_merge":
        a = torch.load(os.path.join(OUT, "filtered_s_ar1.pt"), weights_only=False)
        b = torch.load(os.path.join(OUT, "filtered_s_ar1_part.pt"), weights_only=False)
        assert a["sd_digest"] == b["sd_digest"] and a["tau"] == b["tau"] and a["block"] == b["block"]
        assert not (set(a["picks"]) & set(b["picks"]))
        a["picks"] = a["picks"] + b["picks"]
        for k in ("ids", "logits", "margins"):
            a[k] = torch.cat([a[k], b[k]])
        a["candidates"] += b["candidates"]
        a["acceptance_rate"] = len(a["picks"]) / a["candidates"]
        torch.save(a, os.path.join(OUT, "filtered_s_ar1.pt"))
        os.remove(os.path.join(OUT, "filtered_s_ar1_part.pt"))
        print("merged:", len(a["picks"]), "picks of", a["candidates"], "candidates")
    elif len(sys.argv) > 1 and sys.argv[1] == "filtered":
        # 176 blocks of 256 candidates: ~0.25 % pass the margin filter at full length (a property of the near-flat random-init
        # logits, not of the engine) -> >= 100 accepted sequences; ~25 CPU-minutes on 8 cores
        make_filtered("filtered_s_ar1", "parseq", 0, True, 1, None, int(os.environ.get("FILTERED_BLOCKS", "176")), 256, 0.02)
        make_filtered("filtered_s_ar1_len5", "parseq", 0, True, 1, 5, 2, 256, 0.02)
        make_filtered("filtered_ti_ar1_len5", "parseq-tiny", 2, True, 1, 5, 4, 256, 0.012)
    else:
        main()
