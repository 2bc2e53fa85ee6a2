"""TEST INFRASTRUCTURE ONLY — CPU oracle for the SPH_SM_monodomain step.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference`` legs
may import this package.  The product (``sph_sm_monodomain_b200``) never does.

Two back ends with one interface (:class:`CpuSim`):

* ``"port"``  — ``oracle/sphsm_oracle.c``, the in-repo plain-C restatement (always available; built by
  ``make -C oracle oracle`` / ``__graft_entry__.build()``).
* ``"ref"``   — ``oracle/_ref/libsphsm_ref.so``, the GENUINE reference class compiled from the checkout of its
  sources that ``$SPHSM_REFERENCE_DIR`` names, by ``make -C oracle ref`` (git-ignored; only where those sources exist).
  ``"ref_ofast"`` is the same with the reference Makefile's ``-Ofast``.
"""
from .cpu_sim import CpuSim, PARTICLE_DTYPE, available_backends, build_oracle, lib_path  # noqa: F401
