"""TEST INFRASTRUCTURE — not product code.

CPU oracle for the E2FGVI InpaintGenerator.forward hot path.  Only ``tests/``, ``__graft_entry__.smoke()`` and
``bench.py``'s CPU-baseline legs may import this package; the product (``e2fgvi_b200``) never does and has no
CPU fallback.

* ``restate.py``          plain-PyTorch CPU restatement of the reference algorithm (each function cites the
                          reference file:line it follows); dtype-generic (fp32 / fp64).
* ``reference_loader.py`` imports the UNMODIFIED reference from /root/reference through ``mmcv_shim`` (this
                          container only; the GPU box has no /root/reference) to pin the restatement and to
                          generate ``tests/golden``.
* ``gen_golden.py``       the committed script that produced ``tests/golden/*.pt``.

Parity pinning: the reference ships no tests or golden vectors (SURVEY §4).  The restatement is pinned against
outputs of the reference itself, stored as the committed goldens (``gen_golden.py``, ``gen_golden_video.py``), so the
tests need no copy of the reference.  The one third-party op on the path, ``mmcv.ops.modulated_deform_conv2d``
(mmcv-full 1.4.8, environment.yml:135), is NOT installable offline: its stand-in is
``torchvision.ops.deform_conv2d`` (same DCNv2 lineage) and the explicit restatement in ``restate.py`` matches it
bit-for-bit on random inputs — so parity AT THE MMCV BOUNDARY IS UNPINNED against mmcv itself.
"""
