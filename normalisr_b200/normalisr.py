"""Drop-in namespace for the hot path: ``import normalisr_b200.normalisr as norm`` then
``norm.coex(dt, dc)`` / ``norm.de(dg, dt, dc)`` exactly as with
``import normalisr.normalisr as norm`` (reference src/normalisr/normalisr.py:3-9).
Provided here: the association-testing entry points ``coex`` / ``de``, their consumer ``binnet`` and
the steps upstream, ``lcpm``, ``compute_var`` and ``normvar``.  The remaining names of the reference
module (``qc_reads``, ``qc_outlier``, ``scaling_factor``, ``normcov``, ``gotop``, ``pccovt``) are outside
the hot path (SURVEY.md 8) and stay with the reference package; their output feeds these functions
unchanged.  numpy in -> numpy out, always float64 (the reference keeps the input dtype for ``de``, which
this package does as well, and computes everything else in float64 anyway); CUDA tensors in -> CUDA
tensors out.

Beyond the reference's names: ``coexnet(dt, dc, qcut)``, the reference's ``coex`` -> ``binnet`` pipeline
(``cmd_coex.sh``) as one call that keeps P and dot on the GPUs, and ``binnet(..., sparse=True)``, the network in
CSR form, and ``coextop(dt, dc, k)``, every gene's k strongest partners by r^2 without a genes x genes matrix
(on one GPU, or with ``devices=`` on several, bit-identical).
``coexnet`` and ``coextop`` are importable from here but not listed in ``__all__``, which keeps the reference's
names."""
from .binnet import binnet
from .coex import coex, coexnet, coextop  # noqa: F401 - coexnet, coextop: extensions, see above
from .de import de
from .lcpm import lcpm
from .norm import compute_var, normvar

__all__ = ["coex", "de", "binnet", "normvar", "lcpm", "compute_var"]
