"""Test-only import shim that lets the UNMODIFIED reference sources (a checkout of Bostanabad-Research-Group/GP-Plus,
not part of this repository) execute without gpytorch / botorch.  The checkout is looked for in ``$GPPLUS_REFERENCE``,
else in ``oracle/_ref`` (git-ignored); without one the live tests skip and the stored fixtures stand in for it.

TEST INFRASTRUCTURE -- only ``tests/`` and ``tests/golden/make_reference_fixtures.py`` use it; the product package
never imports it, and nothing of the reference is copied: ``install()`` registers a package called ``gpplus``
whose ``__path__`` is the reference checkout itself, so ``import gpplus.models`` runs the reference's own files where
they lie.

What the reference needs and this image lacks:

* ``gpytorch`` / ``botorch`` (not installed, not vendored, no version pinned by the reference; call sites imply
  gpytorch <= 1.9 / botorch <= 0.7, SURVEY.md section 8c).  ``oracle/_ref_shim/gpytorch`` is a dense-torch
  re-statement of the part of gpytorch's public API the reference's hot path touches (Module / priors /
  constraints, Kernel + RBF / Matern / Scale / Product kernels with ``covar_dist``, means, Gaussian likelihoods,
  ``MultivariateNormal.log_prob`` through ``psd_safe_cholesky``, ``ExactGP`` train / eval calls with the exact
  Cholesky prediction strategy).  It is written from the published gpytorch 1.8/1.9 semantics (SURVEY Appendix A),
  NOT copied from gpytorch, and is therefore itself unverified third-party semantics -- what it pins is every line
  of GP+'s OWN code on the path (model construction, one-hot / zeta tables, latent map, kernel tree, means, noise
  model, MLLObjective packing, priors, bounds, multi-start fit, predict, acquisition functions).
  ``botorch`` is only imported for base classes and a posterior wrapper: stubs.
* ``turtle`` (``from turtle import forward`` at likelihoods_noise/multifidelity.py:16 needs tkinter),
  ``matplotlib``, ``sobol_seq``: stubs.
"""
import importlib.machinery
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
REFERENCE = os.environ.get("GPPLUS_REFERENCE", os.path.join(os.path.dirname(HERE), "_ref"))


def available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE, "models"))


def install():
    """Make ``import gpplus`` resolve to the reference checkout and ``import gpytorch`` to the shim."""
    if not available():
        raise RuntimeError("reference checkout not found at %s" % REFERENCE)
    if HERE not in sys.path:
        sys.path.insert(0, HERE)  # gpytorch, botorch, turtle, matplotlib, sobol_seq stubs
    if "gpplus" not in sys.modules:
        pkg = types.ModuleType("gpplus")
        pkg.__path__ = [REFERENCE]
        pkg.__spec__ = importlib.machinery.ModuleSpec("gpplus", None, is_package=True)
        pkg.__spec__.submodule_search_locations = [REFERENCE]
        sys.dont_write_bytecode = True  # leave the reference checkout as it is
        sys.modules["gpplus"] = pkg
    import gpytorch  # noqa: F401  (the shim)
    return sys.modules["gpplus"]
