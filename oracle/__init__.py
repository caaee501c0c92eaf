"""CPU oracle for the gradient-weighted attention-relevancy path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` is part of the product: only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs may import
it, and there only as the checker (or as the timed CPU baseline), never as the thing shipped.  The
product path (``transformer-mm-explainability_b200``) never imports this package and fails loudly when
its CUDA library is missing.

Parity status: the reference ships NO tests / golden vectors for the relevancy path (SURVEY.md §4), so
the oracle is pinned against *outputs of the reference itself run in the build container*:
``oracle/make_golden.py`` imports the unmodified reference from ``/root/reference`` (with the import shims
of ``oracle/ref_shims.py``), runs it on seeded inputs and commits the results under ``tests/golden/``.
``tests/test_oracle_golden.py`` checks this restatement against those fixtures everywhere, and
``tests/test_oracle_vs_reference.py`` at wider shapes (ViT-B/32 full size; fixture ``oracle_vs_reference.npz``).
Nothing on the path is unpinned any more (round 2): the ViT-B/16 *model* forward - whose source is not
vendored in the reference tree, SURVEY.md §8c - is pinned against torchvision's ``VisionTransformer`` with shared weights
(``tests/test_vit_pin.py``: logits and every block's attention probabilities), the VisualBERT *embeddings* run the
reference's own ``BertVisioLinguisticEmbeddings`` class loaded by file path (``ref_visualbert._import_embeddings``), and
the LXMERT perturbation loops are the UNMODIFIED reference functions driven with a duck-typed ``self``
(``ref_perturbation``; golden ``tests/golden/lxmert_perturbation.npz``).  VisualBERT's evaluation loop (it needs the mmf
registry and COCO files) is checked against the oracle restatement only; the model it calls is pinned.

Modules: ``rules`` (rules 5-11, rollout, Otsu masks), ``clip_oracle``, ``vit_oracle``, ``detr_oracle``,
``lxmert_oracle``, ``visualbert_oracle`` (forward + generators + baselines + ablations + perturbation steps), ``lrp``
(the relprop sweep behind ``use_lrp=True``; the product's device sweep - ``csrc/lrp.cu`` - is tested against it),
``ref_shims`` / ``ref_detr`` / ``ref_lxmert`` / ``ref_visualbert`` / ``ref_perturbation`` (harnesses that run the unmodified reference on CPU),
``make_golden`` (writes ``tests/golden/*.npz`` from them).  The synthetic workload generators live in the product
package (``mmx_b200/synthetic.py``) and are re-exported by ``clip_oracle`` so both sides see the same tensors.
"""
