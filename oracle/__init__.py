"""CPU oracle for the DotaClient optimizer hot path.

THIS PACKAGE IS TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline /
``--impl reference`` legs may import anything from here.  The product package
``dotaclient_b200`` never imports ``oracle`` and has no CPU fallback: it fails
loudly when the CUDA extension is missing.

Parity status: the reference (TimZaman/dotaclient @ 8615b90) ships NO tests,
golden vectors or fixtures for this path (SURVEY.md section 4), so the oracle is
pinned against *outputs of the reference itself run in the build container*
(``oracle/reference_shim.py`` imports ``/root/reference`` in place; the script
``tests/golden/make_golden.py`` records its outputs as committed fixtures, which
``tests/test_oracle.py`` checks the oracle against bit for bit).  The arithmetic
itself lives in third-party, un-vendored dependencies of the reference
(torch==1.0.0, scipy==1.2.0 -- ``docker/Dockerfile:17-19``); the versions available here are torch 2.11 and
scipy 1.18, which is the only executable truth (drift documented in DESIGN.md).

Modules
-------
ref_policy      parametrised restatement of ``policy.py:36-178`` (hidden_size, cell)
ref_optimizer   restatement of ``optimizer.py:53-64, 328-430, 581-695``
ref_distributed restatement of ``distributed.py:16-79`` semantics (gloo, CPU)
gae_ref.c       plain-C restatement of ``optimizer.py:53-64`` (built by oracle/Makefile)
reference_shim  imports the real reference from /root/reference (build container only)
"""
