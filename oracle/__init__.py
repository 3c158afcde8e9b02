"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the reference ViT forward.

Nothing under ``oracle/`` is part of the product path.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline / ``--impl
reference`` legs may import it, and there only as the checker or the timed
CPU baseline, never as a fallback for the CUDA path.

PARITY: pinned to a run of the reference's OWN SOURCE, not to a run of its libraries.  jax / jaxlib / flax are
absent and not installable here and the reference ships no tests, golden vectors or fixtures (SURVEY.md section 8c), so
the reference's ``vit_flax/vit.py`` and ``simple_vit.py`` are executed UNMODIFIED over ``oracle/flax_shim`` -- a numpy
restatement of the jax / flax.linen API subset they call (third-party dependency, flax 0.5.0 / jax 0.3.13 per the
reference README; the shim's README lists every restated definition).  ``tests/golden/make_reference_golden.py`` stores
what the reference computes (logits on three configs, the dropped forward, ``init`` leaf names / shapes, the printed
output of its demo blocks) as ``tests/golden/ref_*.npz``; ``tests/test_reference_run.py`` holds both oracles and the
CUDA path to those vectors, and re-runs the reference live wherever VIT_FLAX_REFERENCE names it.  So every line written IN
the reference is pinned; what stays restated-not-run is the inside of nn.Dense / nn.LayerNorm / nn.gelu / nn.softmax /
nn.Dropout and Flax's auto-naming, cross-checked by two independent restatements (numpy float64 in ``vit_numpy.py``,
torch-CPU float32 in ``vit_torch.py``), an einops check of the patchify order, the known answers the reference documents
(output shape ``(1, 1000)`` -- README.md:34 -- and the parameter count its demo prints), and a third-party
implementation of the same architecture (HuggingFace ``transformers`` ViTForImageClassification, configured like vit.py
and loaded through an explicit weight-layout mapping) that reproduces the oracle's logits to 1e-10 in float64
(tests/test_oracle.py).
"""
