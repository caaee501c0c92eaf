"""Generate the committed golden fixtures under ``tests/golden/`` by running the UNMODIFIED reference.

TEST INFRASTRUCTURE ONLY.  Run in the build container (needs ``/root/reference``)::

    python -m oracle.make_golden

The reference ships no known-answer tests for the relevancy path (SURVEY.md §4), so these fixtures - outputs of
the reference's own code on seeded inputs - are what pins the oracle restatement (and, through it, the CUDA
engine).  Fixtures hold inputs, weights (tiny configs only) and the reference outputs, so they can be checked
on the GPU box where the reference tree does not exist.
"""
from __future__ import annotations

import importlib.util
import os

import numpy as np
import torch

from . import clip_oracle as co
from . import ref_shims as rs

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def _load_module(name, relpath):
    spec = importlib.util.spec_from_file_location(name, os.path.join(rs.REFERENCE_ROOT, relpath))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def golden_clip(tag, cfg, batch, wseed, iseed):
    sd = co.init_state_dict(cfg, seed=wseed)
    images, tokens = co.synthetic_inputs(cfg, batch, seed=iseed)
    model = rs.build_reference_clip(cfg, sd)
    out = {"cfg": np.array(cfg.ref_args(), dtype=np.int64), "images": images.numpy(), "tokens": tokens.numpy()}
    for k, v in sd.items():
        out["sd." + k] = v.numpy()
    for sl in (-1, 0, 1):
        # B distinct images == per-sample calls of the reference (its interpret() repeats ONE image,
        # CLIP_explainability.ipynb:153; samples are independent because only diag logits are summed, :156-160)
        rts, ris = [], []
        for b in range(batch):
            rt, ri = rs.reference_interpret(images[b:b + 1], tokens[b:b + 1], model, "cpu", sl, sl)
            rts.append(rt.detach())
            ris.append(ri.detach())
        out[f"distinct.sl{sl}.R_text"] = torch.cat(rts).numpy()
        out[f"distinct.sl{sl}.R_image"] = torch.cat(ris).numpy()
        rt, ri = rs.reference_interpret(images[:1], tokens, model, "cpu", sl, sl)
        out[f"repeat.sl{sl}.R_text"] = rt.detach().numpy()
        out[f"repeat.sl{sl}.R_image"] = ri.detach().numpy()
    lpi, _ = model(images, tokens)      # hooks need grad mode (CLIP/clip/auxilary.py:250)
    out["logits_per_image"] = lpi.detach().numpy()
    np.savez_compressed(os.path.join(OUT, f"clip_{tag}.npz"), **out)
    print("wrote", tag, {k: v.shape for k, v in out.items() if not k.startswith("sd.")})


def golden_clip_example():
    """CLIP/example.py:8-53 (the older interpret: one image, N texts, ``index``, all image blocks) run unmodified."""
    cfg = co.EXAMPLE
    sd = co.init_state_dict(cfg, seed=4)
    images, tokens = co.synthetic_inputs(cfg, 3, seed=21)
    model = rs.build_reference_clip(cfg, sd)
    out = {"cfg": np.array(cfg.ref_args(), dtype=np.int64), "image": images[:1].numpy(), "tokens": tokens.numpy()}
    for k, v in sd.items():
        out["sd." + k] = v.numpy()
    for index in (None, 0, 1, 2):
        R, logits = rs.reference_example_interpret(images[:1], tokens, model, "cpu", index)
        out[f"R.index{index}"] = R.numpy()
        out["logits_per_image"] = logits.numpy()
    np.savez_compressed(os.path.join(OUT, "clip_example.npz"), **out)
    print("wrote clip_example", {k: v.shape for k, v in out.items() if not k.startswith("sd.")})


def golden_lxmert_perturbation():
    """lxmert/lxmert/perturbation.py:85-194 (the two perturbation loops, unmodified source) on one synthetic item; the model
    behind ``self.lxmert_vqa`` is the unmodified reference LXMERT (ref_lxmert)."""
    from . import lxmert_oracle as lo, ref_lxmert, ref_perturbation as rp
    cfg = lo.LXMERT_TINY
    sd = lo.init_state_dict(cfg, 3)
    ids, feats, boxes = lo.synthetic_inputs(cfg, 1, 9, 11, seed=6)
    rtt, rti = ref_lxmert.generate_ours(cfg, sd, ids, feats, boxes, use_lrp=False)
    cam_image, cam_text = rti[0][0].clone(), rtt[0][0].clone()          # perturbation.py:241-244: row of [CLS]
    model_fn = ref_lxmert.forward_fn(cfg, sd)
    out = {"ids": ids.numpy(), "feats": feats.numpy(), "boxes": boxes.numpy(), "cam_image": cam_image.numpy(),
           "cam_text": cam_text.numpy()}
    for k, v in sd.items():
        out["sd." + k] = v.numpy()
    for modality in ("image", "text"):
        for positive in (False, True):
            scores, steps = rp.run(model_fn, ids, feats, boxes, cam_image, cam_text, modality, positive, cfg.num_labels)
            out[f"scores.{modality}.{int(positive)}"] = scores.numpy()
    out["pert_steps"] = np.array(steps)
    np.savez_compressed(os.path.join(OUT, "lxmert_perturbation.npz"), **out)
    print("wrote lxmert_perturbation", {k: v.shape for k, v in out.items() if not k.startswith("sd.")})


def golden_rules():
    detr = _load_module("ref_detr_eg", "DETR/modules/ExplanationGenerator.py")
    lx = _load_module("ref_lxmert_eg", "lxmert/lxmert/src/ExplanationGenerator.py")
    g = torch.Generator().manual_seed(99)
    out = {}
    H, T, S = 4, 10, 13
    cam_ss = torch.softmax(torch.randn(H, T, T, generator=g), -1)
    grad_ss = torch.randn(H, T, T, generator=g)
    cam_sq = torch.softmax(torch.randn(H, T, S, generator=g), -1)
    grad_sq = torch.randn(H, T, S, generator=g)
    out["cam_ss"], out["grad_ss"], out["cam_sq"], out["grad_sq"] = (x.numpy() for x in (cam_ss, grad_ss, cam_sq, grad_sq))
    abar_ss = detr.avg_heads(cam_ss, grad_ss)
    abar_sq = lx.avg_heads(cam_sq, grad_sq)
    out["abar_ss"], out["abar_sq"] = abar_ss.numpy(), abar_sq.numpy()
    # relevancy state after one self-attention update (so that R-I has a positive diagonal, as in the path)
    R_ss = torch.eye(T) + abar_ss
    R_qq = torch.eye(S) + detr.avg_heads(torch.softmax(torch.randn(H, S, S, generator=g), -1),
                                         torch.randn(H, S, S, generator=g))
    R_sq = 0.1 * torch.rand(T, S, generator=g)
    R_qs = 0.1 * torch.rand(S, T, generator=g)
    out["R_ss"], out["R_qq"], out["R_sq"], out["R_qs"] = (x.numpy() for x in (R_ss, R_qq, R_sq, R_qs))
    a, b = detr.apply_self_attention_rules(R_ss, R_sq, abar_ss)
    out["self.R_ss_add"], out["self.R_sq_add"] = a.numpy(), b.numpy()
    out["hr.R_ss"] = detr.handle_residual(R_ss).numpy()
    out["hr.R_qq"] = lx.handle_residual(R_qq).numpy()
    for norm in (True, False):
        for self10 in (True, False):
            key = f"n{int(norm)}s{int(self10)}"
            out[f"mm_detr.{key}"] = detr.apply_mm_attention_rules(
                R_ss, R_qq, abar_sq.clone(), apply_normalization=norm, apply_self_in_rule_10=self10).numpy()
            x, y = lx.apply_mm_attention_rules(R_ss, R_qq, R_qs, abar_sq.clone(), apply_normalization=norm,
                                               apply_self_in_rule_10=self10)
            out[f"mm_lx.{key}.sq"], out[f"mm_lx.{key}.ss"] = x.numpy(), y.numpy()
    # NaN -> 0 guard (DETR only): a state with an all-zero R-I row gives 0/0 in handle_residual
    out["mm_detr.identity_state"] = detr.apply_mm_attention_rules(torch.eye(T), torch.eye(S), abar_sq.clone()).numpy()
    mats = [torch.softmax(torch.randn(T, T, generator=g), -1) for _ in range(5)]
    out["rollout.mats"] = torch.stack(mats).numpy()
    for sl in (0, 2):
        out[f"rollout.sl{sl}"] = detr.compute_rollout_attention([m.clone() for m in mats], sl).numpy()
    np.savez_compressed(os.path.join(OUT, "rules.npz"), **out)
    print("wrote rules", len(out))


def golden_detr():
    from . import detr_oracle as do, ref_detr
    cfg = do.DETR_TINY
    sd = do.init_state_dict(cfg, 5)
    src, pos, tq = do.synthetic_inputs(cfg, 3, 3, 4, seed=1)
    out = {"cfg": np.array([cfg.d_model, cfg.nhead, cfg.enc_layers, cfg.dec_layers, cfg.dim_ff, cfg.queries, cfg.classes]),
           "src": src.numpy(), "pos": pos.numpy(), "tq": tq.numpy()}
    for k, v in sd.items():
        out["sd." + k] = v.numpy()
    for norm in (True, False):
        for s10 in (True, False):
            r = ref_detr.generate_ours(cfg, sd, src, pos, tq, normalize_self_attention=norm, apply_self_in_rule_10=s10)
            out[f"R.n{int(norm)}s{int(s10)}"] = r.numpy()
    for method in ("raw_attn", "rollout", "attn_gradcam"):          # baselines behind the same API (SURVEY.md §8f-2)
        out["base." + method] = ref_detr.generate_baseline(cfg, sd, src, pos, tq, method).numpy()
    for norm in (True, False):                                   # use_lrp=True (the reference default): target for §8f-4
        for s10 in (True, False):
            out[f"R.lrp.n{int(norm)}s{int(s10)}"] = ref_detr.generate_ours(cfg, sd, src, pos, tq, use_lrp=True, normalize_self_attention=norm,
                                                                         apply_self_in_rule_10=s10).numpy()
    for name, cam in ref_detr.lrp_attn_cams(cfg, sd, src[:1], pos[:1], int(tq[0])).items():
        out["lrp.cam." + name] = cam.numpy()                     # per-layer LRP relevance of A, sample 0 (debugging aid)
    for name, cam in ref_detr.lrp_attn_cams(cfg, sd, src[:1], pos[:1], int(tq[0]), double=True).items():
        out["lrp.cam64." + name] = cam.numpy()                   # the same from the reference run in float64
    for method in ("transformer_att", "partial_lrp"):               # the LRP-based baselines (EG:64-108, :197-224)
        out["base." + method] = ref_detr.generate_baseline(cfg, sd, src, pos, tq, method).numpy()
    out["abl.noagg"] = ref_detr.generate_ours_abl(cfg, sd, src, pos, tq).numpy()    # GeneratorAlbationNoAgg (EG:306-403)
    out["abl.noagg.s0"] = ref_detr.generate_ours_abl(cfg, sd, src, pos, tq, apply_self_in_rule_10=False).numpy()
    np.savez_compressed(os.path.join(OUT, "detr_tiny.npz"), **out)
    print("wrote detr_tiny", out["R.n1s1"].shape)


def golden_lxmert():
    from . import lxmert_oracle as lo, ref_lxmert
    cfg = lo.LXMERT_TINY
    sd = lo.init_state_dict(cfg, 3)
    ids, feats, boxes = lo.synthetic_inputs(cfg, 3, 6, 5, seed=2)
    out = {"ids": ids.numpy(), "feats": feats.numpy(), "boxes": boxes.numpy()}
    for k, v in sd.items():
        out["sd." + k] = v.numpy()
    for norm in (True, False):
        for s10 in (True, False):
            rtt, rti = ref_lxmert.generate_ours(cfg, sd, ids, feats, boxes, normalize_self_attention=norm,
                                                apply_self_in_rule_10=s10)
            out[f"Rtt.n{int(norm)}s{int(s10)}"], out[f"Rti.n{int(norm)}s{int(s10)}"] = rtt.numpy(), rti.numpy()
    for method in ("raw_attn", "rollout", "attn_gradcam"):
        rtt, rti = ref_lxmert.generate_baseline(cfg, sd, ids, feats, boxes, method)
        out[f"base.{method}.Rtt"], out[f"base.{method}.Rti"] = rtt.numpy(), rti.numpy()
    for norm in (True, False):                                   # use_lrp=True (the reference default): target for §8f-4
        for s10 in (True, False):
            rtt, rti = ref_lxmert.generate_ours(cfg, sd, ids, feats, boxes, use_lrp=True, normalize_self_attention=norm,
                                                apply_self_in_rule_10=s10)
            out[f"Rtt.lrp.n{int(norm)}s{int(s10)}"], out[f"Rti.lrp.n{int(norm)}s{int(s10)}"] = rtt.numpy(), rti.numpy()
    for method in ("transformer_attr", "partial_lrp"):              # the LRP-based baselines (EG:373-507)
        rtt, rti = ref_lxmert.generate_baseline(cfg, sd, ids, feats, boxes, method)
        out[f"base.{method}.Rtt"], out[f"base.{method}.Rti"] = rtt.numpy(), rti.numpy()
    rtt, rti = ref_lxmert.generate_ours_no_agg(cfg, sd, ids, feats, boxes, normalize_self_attention=False)   # EG:215-365
    out["abl.noagg.Rtt"], out["abl.noagg.Rti"] = rtt.numpy(), rti.numpy()
    np.savez_compressed(os.path.join(OUT, "lxmert_tiny.npz"), **out)
    print("wrote lxmert_tiny", out["Rtt.n1s1"].shape, out["Rti.n1s1"].shape)


def golden_otsu():
    """cv2.threshold(THRESH_BINARY + THRESH_OTSU) itself on seeded maps, through the exact expression of
    DETR/mask_generator.py:115-121."""
    import cv2
    rng = np.random.default_rng(0)
    maps, n = [], 625
    for t in range(48):
        kind = t % 4
        if kind == 0:
            x = rng.random(n)
        elif kind == 1:
            x = rng.random(n) ** 6
        elif kind == 2:
            x = np.concatenate([rng.normal(0.2, 0.05, n // 2), rng.normal(0.8, 0.1, n - n // 2)])
        else:
            x = rng.integers(0, 3, n).astype(np.float64)
        maps.append(x.astype(np.float32))
    cams = torch.tensor(np.stack(maps))
    masks, ths = [], []
    for cam in cams:
        c = (cam - cam.min()) / (cam.max() - cam.min()) * 255
        img = c.reshape(25, 25).data.cpu().numpy().astype(np.uint8)
        ret, th = cv2.threshold(img, 0, 255, cv2.THRESH_BINARY + cv2.THRESH_OTSU)
        masks.append(th.reshape(-1).astype(np.float32)); ths.append(int(ret))
    np.savez_compressed(os.path.join(OUT, "otsu.npz"), cams=cams.numpy(), masks=np.stack(masks), thresholds=np.array(ths),
                        cv2_version=np.array(cv2.__version__))
    print("wrote otsu", len(ths), "cv2", cv2.__version__)


def golden_visualbert():
    from . import visualbert_oracle as vo, ref_visualbert
    cfg = vo.VISUALBERT_TINY
    sd = vo.init_state_dict(cfg, 3)
    inp = vo.synthetic_inputs(cfg, 3, 7, 6, seed=4)
    inp["attention_mask"][1, -2:] = 0                     # sample 1: two padded boxes (image_mask, visual_bert.py:548-555)
    out = {"inp." + k: v.numpy() for k, v in inp.items()}
    for k, v in sd.items():
        out["sd." + k] = v.numpy()
    for method in ("ours", "raw_attn", "rollout", "attn_gradcam"):
        out["R." + method] = ref_visualbert.generate(cfg, sd, inp, method).numpy()
    out["R.ours.index5"] = ref_visualbert.generate(cfg, sd, inp, "ours", index=5).numpy()
    out["R.rollout.sl1"] = ref_visualbert.generate(cfg, sd, inp, "rollout", start_layer=1).numpy()
    out["R.transformer_att"] = ref_visualbert.generate(cfg, sd, inp, "transformer_att").numpy()        # LRP-based (§8f-4 targets)
    out["R.transformer_att.sl1"] = ref_visualbert.generate(cfg, sd, inp, "transformer_att", start_layer=1).numpy()
    out["R.partial_lrp"] = ref_visualbert.generate(cfg, sd, inp, "partial_lrp").numpy()
    np.savez_compressed(os.path.join(OUT, "visualbert_tiny.npz"), **out)
    print("wrote visualbert_tiny", out["R.ours"].shape)


def golden_vs_reference():
    """The cases of tests/test_oracle_vs_reference.py at shapes wider than the fixtures above (ViT-B/32 full size, a
    VisualBERT / DETR / LXMERT wider than the tiny configs).  Weights and inputs come from the seeded generators the test
    calls again, so only the reference outputs are stored."""
    from . import detr_oracle as do, lxmert_oracle as lo, visualbert_oracle as vo, ref_detr, ref_lxmert, ref_visualbert
    out = {}
    cfg = co.VIT_B32
    sd = co.init_state_dict(cfg, seed=0)
    images, tokens = co.synthetic_inputs(cfg, 2, seed=7)
    model = rs.build_reference_clip(cfg, sd)
    for sl in (-1, 0):
        rts, ris = [], []
        for b in range(2):
            rt, ri = rs.reference_interpret(images[b:b + 1], tokens[b:b + 1], model, "cpu", sl, sl)
            rts.append(rt.detach())
            ris.append(ri.detach())
        out[f"vit_b32.sl{sl}.R_text"], out[f"vit_b32.sl{sl}.R_image"] = torch.cat(rts).numpy(), torch.cat(ris).numpy()
    del model, sd
    cfg = co.SMALL
    sd = co.init_state_dict(cfg, seed=4)
    images, tokens = co.synthetic_inputs(cfg, 5, seed=9)
    rt, ri = rs.reference_interpret(images[:1], tokens, rs.build_reference_clip(cfg, sd), "cpu", 0, 0)
    out["repeat_small.R_text"], out["repeat_small.R_image"] = rt.detach().numpy(), ri.detach().numpy()
    cfg = vo.VisualBertConfig(hidden=128, heads=8, intermediate=256, layers=4, vocab=80, max_pos=32, visual_dim=48, num_labels=31)
    sd = vo.init_state_dict(cfg, 11)
    inp = vo.synthetic_inputs(cfg, 2, 9, 12, seed=5)
    for method in ("ours", "raw_attn", "rollout", "attn_gradcam"):
        out["visualbert." + method] = ref_visualbert.generate(cfg, sd, inp, method).numpy()
    cfg = do.DetrConfig(128, 4, 3, 3, 192, 9, 6)
    sd = do.init_state_dict(cfg, 9)
    src, pos, tq = do.synthetic_inputs(cfg, 2, 5, 6, seed=4)
    out["detr_lrp"] = ref_detr.generate_ours(cfg, sd, src, pos, tq, use_lrp=True, normalize_self_attention=False).numpy()
    cfg = lo.LxmertConfig(hidden=128, heads=4, intermediate=160, l_layers=3, x_layers=3, r_layers=2, vocab=70, max_pos=20,
                          feat_dim=40, pos_dim=4, num_labels=17)
    sd = lo.init_state_dict(cfg, 6)
    ids, feats, boxes = lo.synthetic_inputs(cfg, 2, 9, 7, seed=3)
    rtt, rti = ref_lxmert.generate_ours(cfg, sd, ids, feats, boxes, use_lrp=True)
    out["lxmert_lrp.Rtt"], out["lxmert_lrp.Rti"] = rtt.numpy(), rti.numpy()
    np.savez_compressed(os.path.join(OUT, "oracle_vs_reference.npz"), **out)
    print("wrote oracle_vs_reference", {k: v.shape for k, v in out.items()})


def main():
    os.makedirs(OUT, exist_ok=True)
    argv = __import__("sys").argv
    if "--vs-reference" in argv:
        golden_vs_reference()
        return
    if "--visualbert" in argv:
        golden_visualbert()
        return
    if "--otsu" in argv:
        golden_otsu()
        return
    if "--clip-example" in argv:
        golden_clip_example()
        return
    if "--lxmert-perturbation" in argv:
        golden_lxmert_perturbation()
        return
    if "--only-new" in argv:
        golden_detr()
        golden_lxmert()
        golden_visualbert()
        return
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    golden_rules()
    golden_clip("tiny", co.TINY, 3, wseed=1, iseed=7)
    golden_clip("small", co.SMALL, 4, wseed=2, iseed=11)
    golden_clip_example()
    golden_detr()
    golden_lxmert()
    golden_lxmert_perturbation()
    golden_visualbert()
    golden_otsu()
    golden_vs_reference()


if __name__ == "__main__":
    main()
