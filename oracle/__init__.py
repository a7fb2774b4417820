"""CPU oracle for the DynaBOA hot path -- TEST INFRASTRUCTURE ONLY.

This package restates, on CPU in plain torch (fp32 by default, fp64 on request), the
algorithm of the reference's per-frame hot path (SURVEY.md §8):

* ``geometry_ref``  -- reference utils/geometry.py (rot6d, quaternion Rodrigues,
                       rotation-matrix -> axis-angle, perspective projection)
* ``prior_ref``     -- reference utils/smplify/prior.py:181-196 (merged max-mixture NLL)
* ``hmr_ref``       -- reference model/hmr.py (GroupNorm ResNet-50 + iterative regressor)
* ``smplx_ref``     -- third-party ``smplx`` (version unpinned in reference requirements.txt:22):
                       SMPL.forward / lbs / vertex_joint_selector + reference model/smpl.py wrapper
* ``l2l_ref``       -- third-party ``learn2learn==0.1.5`` (reference requirements.txt:10):
                       MAML.clone / MAML.adapt, first-order
* ``adaptor_ref``   -- reference base_adaptor.py losses/adaptation + dynaboa_benchmark.py
                       ``Adaptor.adaptation`` / ``inference`` orchestration
* ``eval_ref``      -- reference dynaboa_benchmark.py:217-240 + utils/pose_utils.py:9-64 (H36M joints, MPJPE,
                       Procrustes PA-MPJPE, PVE), pinned against the reference's own numpy Procrustes

Pinning status (see DESIGN.md "Oracle"):

* geometry / prior / hmr restatements are checked bit-for-bit against the reference's own
  modules imported from the checkout named by DBOA_REFERENCE_ROOT by ``oracle/make_golden.py``,
  and the resulting vectors are committed under ``tests/golden/``.
* the loss assembly and the adaptation orchestration are checked against the reference's own
  ``base_adaptor.BaseAdaptor`` / ``dynaboa_benchmark.Adaptor`` code executed on CPU with the two
  missing third-party packages replaced by the restatements here.
* smplx and learn2learn themselves are NOT available offline (no network, not vendored):
  **parity unpinned** for those two restatements -- they follow the published upstream
  algorithm (SURVEY.md Appendix A/B) and analytic properties only.

Only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` / ``--impl reference``
legs of ``bench.py`` may import this package, and only as the checker / timed CPU baseline.
The product package ``dynaboa_b200`` never imports it and has no CPU fallback.
"""
