"""CPU oracle for the WaterNet hot path -- TEST INFRASTRUCTURE ONLY.

This package restates, on the CPU, the algorithms of the reference
(tnwei/waternet @ 2091896):

* ``oracle.preprocess`` -- ``waternet/data.py`` (white balance, gamma, Lab+CLAHE
  histogram equalisation) in plain numpy, including the OpenCV 4.x 8-bit fixed
  point RGB<->Lab conversion and CLAHE that ``data.py:68-78`` delegates to cv2.
* ``oracle.forward`` -- ``waternet/net.py`` (confidence-map generator, three
  refiners, gated sum) as a functional torch-CPU fp32/fp64 evaluation, and its float64
  gradients (``waternet_grads``, CPU or GPU) as the ground truth of the backward tests.

Only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` /
``--impl reference`` legs of ``bench.py`` may import this package, and only as
the checker / the timed CPU baseline.  Nothing under ``waternet_b200/`` imports
it; the product path fails loudly when the CUDA library is missing.

Parity pin: the reference holds no golden vectors or tests (SURVEY.md section 4).
The oracle is pinned against the reference itself, imported unchanged from
``/root/reference`` in the build container: ``tests/golden/make_golden.py``
writes ``tests/golden/*.npz`` from the reference's own outputs, and
``tests/test_oracle.py`` checks the oracle against those fixtures everywhere and
against the live reference / cv2 where they are importable.
"""
