"""TEST INFRASTRUCTURE ONLY — the CPU oracle for the HuMoR Stage-III hot path.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import anything from this package, and only as the
checker.  The product (``humor_b200``) never imports it and has no CPU fallback.

Contents
  smplh_lbs.py    restatement of smplx==0.1.28 ``lbs`` / ``SMPLH.forward`` (third-party,
                  absent from /root/reference; algorithm from SURVEY.md Appendix A.1 and
                  anchored on the reference's call sites body_model/body_model.py:61-99).
  stage3_port.py  plain-torch restatement of the reference's Stage-III closure
                  (models/humor_model.py, fitting/motion_optimizer.py, fitting/fitting_loss.py,
                  fitting/fitting_utils.py, utils/transforms.py), every function citing the
                  reference file:line it follows.  Portable: travels to the GPU box.
  ref_import.py   imports the UNMODIFIED reference from /root/reference (this container only)
                  behind a ``smplx`` stub backed by smplh_lbs.py.
  make_golden.py  runs the real reference and writes tests/golden/stage*.npz.
  make_golden_ref.py  runs the real reference on the inputs of the other comparison tests and
                  writes tests/golden/ref_*.npz.

Parity pinning: the reference ships no tests or golden vectors (SURVEY.md §4).  The port is
pinned against the committed fixtures the make_golden*.py scripts generated from the
reference; no test needs the reference itself, so every comparison runs on every machine.
The LBS restatement has no runnable third-party source to check against (smplx is not
installable offline): **LBS parity is pinned only by the analytic known-answer cases** in
tests/test_oracle_lbs.py (zero pose, rigid root rotation, hand-column independence).
"""
