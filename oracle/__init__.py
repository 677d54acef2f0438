"""CPU oracle for the AprilGroup tracking hot path.  TEST INFRASTRUCTURE ONLY.

Nothing under ``oracle/`` is shipped or measured as the product: only
``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` / ``--impl
reference`` legs of ``bench.py`` import it, and only as the checker.

Parity status per stage (see DESIGN.md):
  * APE (detect_pose.py:467-574 + cv2.solvePnP): pinned - ``ape_oracle`` is
    checked against committed golden vectors that the unmodified reference
    generated (``make_golden`` driving it through ``ref_runner``).
  * pyramid / LK: the reference snapshot has no such code; the frozen spec is
    OpenCV 4.13 ``pyrDown`` / ``Scharr`` / ``calcOpticalFlowPyrLK`` (binary in
    this image, third-party, source absent).  ``lk_oracle`` calls it and also
    holds a numpy restatement pinned against it.
  * frame ingest (undistort_frame, detect_pose.py:147-183, + BGR2GRAY,
    detect_pose.py:602): ``undistort_oracle`` restates cv::undistort /
    cv::cvtColor and is pinned bit for bit against the installed cv2, i.e.
    against the calls the reference itself makes.
  * dense pose refinement: no reference code exists; ``dpr_oracle`` IS the
    executable spec.  PARITY UNPINNED against the reference for this stage
    (pinned only against scipy.optimize.least_squares on the same residual).
"""
