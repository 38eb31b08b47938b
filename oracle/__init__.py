"""CPU oracle for the frame-differencing hot loop -- TEST INFRASTRUCTURE ONLY.

This package restates, on the CPU, the arithmetic of the reference's per-frame
loop (frame_differencing.py:85-133, motion_compression_opt.py:84-90,141-185).
It is the checker the CUDA path is compared against.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl
reference`` legs may import it.  Nothing under
``dynamic_video_compression_surveillance_b200/`` imports it, and the product
path raises if the CUDA library is missing rather than falling back to this.

How the oracle is pinned (the reference ships no tests or golden vectors,
SURVEY.md section 4):

* ``oracle/stage_ops.py``  -- closed-form numpy restatements of every cv2 /
  numpy call on the path.  ``tests/test_oracle_vs_cv2.py`` checks each against
  the real ``cv2`` call (opencv-python is the reference's pinned third-party
  dependency, requirements.txt:2 ``==4.11.0.86``; the image has 4.13.0).
* ``oracle/loops.py``      -- the loop bodies restated on arrays.
* ``oracle/flow_ops.py``   -- cv2.calcOpticalFlowFarneback in cv2's scalar
  operation order; ``tests/test_flow_oracle_cpu.py`` checks it against cv2
  byte for byte and ``tests/test_flow_exact_gpu.py`` the kernels against it.
* ``oracle/cv2_proxy.py`` + ``oracle/make_golden.py`` -- run the UNMODIFIED
  reference modules from /root/reference on array-backed VideoCapture /
  VideoWriter fakes (no lossy codec) and commit the outputs as fixtures under
  ``tests/golden/``.  ``tests/test_oracle_golden.py`` checks ``loops.py``
  against those fixtures, so the restatement is pinned to outputs of the
  reference itself.
"""
