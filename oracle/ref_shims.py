"""Import shims that let the UNMODIFIED reference run on CPU in the build container.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).  The reference tree is needed only to regenerate the fixtures
under ``tests/golden/``, so everything here is used by ``oracle/make_golden.py`` and nothing else.
Shims (SURVEY.md §8c):
  * ``ftfy`` stub            - CLIP/clip/simple_tokenizer.py:6 imports it; the tokenizer is never called here.
  * ``Tensor.cuda`` identity - the reference hard-codes ``.cuda()`` (CLIP_explainability.ipynb:160,
                               DETR/modules/ExplanationGenerator.py:160); on CPU it must be a no-op.
"""
from __future__ import annotations

import contextlib
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("MMX_REFERENCE_ROOT", "/root/reference")


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "CLIP", "clip"))


def _ensure_path():
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    if "ftfy" not in sys.modules:
        sys.modules["ftfy"] = types.ModuleType("ftfy")
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)


@contextlib.contextmanager
def cuda_is_identity():
    import torch
    orig = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        yield
    finally:
        torch.Tensor.cuda = orig


def build_reference_clip(cfg, state_dict=None, seed: int = 0):
    """Instantiate the reference ``CLIP`` (CLIP/clip/model.py:248) in fp32 (as ``clip.load`` does on CPU,
    CLIP/clip/clip.py:117-118) and optionally load a state_dict into it."""
    _ensure_path()
    import torch
    from CLIP.clip.model import CLIP
    torch.manual_seed(seed)
    model = CLIP(*cfg.ref_args()).float().eval()
    if state_dict is not None:
        missing, unexpected = model.load_state_dict(state_dict, strict=False)
        assert not unexpected, unexpected
        assert all(m.endswith("attn_mask") for m in missing), missing
    return model


def reference_interpret(image, texts, model, device="cpu", start_layer=-1, start_layer_text=-1):
    """Runs the notebook's ``interpret`` (CLIP_explainability.ipynb cell 6) by exec-ing the cell source straight
    from the reference's .ipynb - nothing is copied into this repo - with ``.cuda()`` made an identity."""
    _ensure_path()
    import json
    import numpy as np
    import torch
    with open(os.path.join(REFERENCE_ROOT, "CLIP_explainability.ipynb")) as f:
        nb = json.load(f)
    src = None
    for cell in nb["cells"]:
        s = "".join(cell["source"])
        if cell["cell_type"] == "code" and s.lstrip().startswith("def interpret("):
            src = s
            break
    assert src is not None, "interpret() cell not found"
    ns = {"torch": torch, "np": np, "start_layer": -1, "start_layer_text": -1}
    exec(compile(src, "CLIP_explainability.ipynb:cell6", "exec"), ns)
    with cuda_is_identity():
        return ns["interpret"](image, texts, model, device, start_layer=start_layer,
                               start_layer_text=start_layer_text)


def reference_example_interpret(image, text, model, device="cpu", index=None):
    """Runs the older ``interpret`` of CLIP/example.py:8-53 (one image, N texts, all image blocks, ``R[0,0] = 0``) by
    exec-ing the function source straight from the reference file.  The function plots and returns nothing; the relevance
    vector is captured where the unmodified code hands it to ``torch.nn.functional.interpolate`` (:42-43).  matplotlib is
    absent in this image and is stubbed (``plt.imshow`` / ``plt.show`` are no-ops); needs a 7x7 patch grid at 224 px
    (hard-coded in :42-43).  Returns (image_relevance [49], logits_per_image [1,N])."""
    _ensure_path()
    import numpy as np
    import torch
    import cv2
    with open(os.path.join(REFERENCE_ROOT, "CLIP", "example.py")) as f:
        src = f.read()
    start, end = src.index("def interpret("), src.index("def main(")
    plt = types.SimpleNamespace(imshow=lambda *a, **k: None, show=lambda *a, **k: None)
    ns = {"torch": torch, "np": np, "cv2": cv2, "plt": plt, "print": lambda *a, **k: None}
    exec(compile(src[start:end], "CLIP/example.py:interpret", "exec"), ns)
    captured = {}
    orig = torch.nn.functional.interpolate

    def spy(x, *a, **k):
        captured["R"] = x.detach().clone().reshape(-1)
        return orig(x, *a, **k)

    torch.nn.functional.interpolate = spy
    try:
        with cuda_is_identity():
            ns["interpret"](image, text, model, device, index)
            logits, _ = model(image, text)
    finally:
        torch.nn.functional.interpolate = orig
    return captured["R"], logits.detach()
