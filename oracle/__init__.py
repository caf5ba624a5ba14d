"""CPU oracle for the panorama -> plane hot path.  TEST INFRASTRUCTURE ONLY.

Nothing under ``oracle/`` is part of the product.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference``
legs may import it, and there only as the checker / the timed CPU baseline.  The product
path (``360-to-planer-images_b200/``) never imports this package and fails loudly when the
CUDA library is missing.

Parity pinning: the reference (``/root/reference/app/panorama_to_plane-pitch.py``) ships no
tests or golden vectors of its own (SURVEY.md section 4), so the oracle is pinned against
outputs of the *unmodified reference executed in the dev container*: ``gen_golden.py`` imports
it by path and stores small input/output vectors under ``tests/golden/`` (library versions
recorded in the fixture).  ``tests/test_oracle_golden.py`` replays them.

Modules
-------
ref_port     two-pass NumPy + cv2.remap restatement (what the reference executes; also the
             timed CPU baseline, ``cpu_baseline.kind == "port"``)
fixedpoint   cv2-free integer model of ``cv2.remap(INTER_LINEAR, BORDER_CONSTANT)`` and the
             single-pass per-pixel restatement the CUDA kernel follows (SURVEY Appendix A)
synth        deterministic synthetic panoramas (noise / smooth / coords)
golden       reads and writes the golden vectors under ``tests/golden/``
"""
