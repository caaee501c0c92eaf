"""CPU: the oracle restatement against outputs of the UNMODIFIED reference at shapes wider than the other goldens
(ViT-B/32 full size, the notebook's repeat mode, VisualBERT / DETR / LXMERT wider than their tiny configs).  The reference
outputs are tests/golden/oracle_vs_reference.npz, written by ``python -m oracle.make_golden --vs-reference``; weights and
inputs come from the same seeded generators here and there, so the fixture holds the reference outputs only."""
import os

import numpy as np
import pytest
import torch

from oracle import clip_oracle as co
from util import rel_err, text_rel_err


@pytest.fixture(scope="module")
def ref(golden_dir):
    return np.load(os.path.join(golden_dir, "oracle_vs_reference.npz"))


@pytest.mark.parametrize("sl", [-1, 0])
def test_vit_b32_full_size(ref, sl):
    cfg = co.VIT_B32
    sd = co.init_state_dict(cfg, seed=0)
    images, tokens = co.synthetic_inputs(cfg, 2, seed=7)
    ot, oi = co.clip_interpret(sd, cfg, images, tokens, sl, sl)
    assert text_rel_err(ot, ref[f"vit_b32.sl{sl}.R_text"]) < 2e-5
    assert rel_err(oi, ref[f"vit_b32.sl{sl}.R_image"]) < 2e-5


def test_repeat_mode_small(ref):
    cfg = co.SMALL
    sd = co.init_state_dict(cfg, seed=4)
    images, tokens = co.synthetic_inputs(cfg, 5, seed=9)
    ot, oi = co.clip_interpret(sd, cfg, images[:1], tokens, 0, 0)
    assert text_rel_err(ot, ref["repeat_small.R_text"]) < 1e-5 and rel_err(oi, ref["repeat_small.R_image"]) < 1e-5


@pytest.mark.parametrize("method", ["ours", "raw_attn", "rollout", "attn_gradcam"])
def test_visualbert_live_reference(ref, method):
    """The unmodified BertEncoder / BertPredictionHeadTransform / SelfAttentionGenerator of the reference at a
    wider shape than the golden file (hidden 128, 8 heads, 4 layers, 9 tokens + 12 boxes)."""
    from oracle import visualbert_oracle as vo
    cfg = vo.VisualBertConfig(hidden=128, heads=8, intermediate=256, layers=4, vocab=80, max_pos=32, visual_dim=48, num_labels=31)
    sd = vo.init_state_dict(cfg, 11)
    inp = vo.synthetic_inputs(cfg, 2, 9, 12, seed=5)
    got = getattr(vo, "generate_" + method)(sd, cfg, inp)
    got = got[0] if isinstance(got, tuple) else got
    assert rel_err(got, ref["visualbert." + method]) < 1e-5


def test_detr_lrp_live_reference_wider(ref):
    """use_lrp=True at a shape other than the golden one (d=128, 4 heads, 3 encoder / 3 decoder layers, 5x6 features,
    9 queries): the restated relprop sweep against the unmodified reference generator."""
    from oracle import detr_oracle as do
    cfg = do.DetrConfig(128, 4, 3, 3, 192, 9, 6)
    sd = do.init_state_dict(cfg, 9)
    src, pos, tq = do.synthetic_inputs(cfg, 2, 5, 6, seed=4)
    got = do.generate_ours_lrp(sd, cfg, src, pos, tq, normalize_self_attention=False)
    assert np.abs(ref["detr_lrp"]).max() > 0
    assert rel_err(got, ref["detr_lrp"]) < 2e-4


def test_lxmert_lrp_live_reference_wider(ref):
    from oracle import lxmert_oracle as lo
    cfg = lo.LxmertConfig(hidden=128, heads=4, intermediate=160, l_layers=3, x_layers=3, r_layers=2, vocab=70, max_pos=20,
                          feat_dim=40, pos_dim=4, num_labels=17)
    sd = lo.init_state_dict(cfg, 6)
    ids, feats, boxes = lo.synthetic_inputs(cfg, 2, 9, 7, seed=3)
    gtt, gti = lo.generate_ours_lrp(sd, cfg, ids, feats, boxes)
    assert rel_err(gtt, ref["lxmert_lrp.Rtt"]) < 1e-5 and rel_err(gti, ref["lxmert_lrp.Rti"]) < 1e-5
