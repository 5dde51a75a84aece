"""Drop-in replacements for the reference's `geometry.gshell_tets` / `geometry.hmsdf_tets_split` modules and its SDF
regulariser `compute_sdf_reg_loss` (geometry/hmsdf.py:162-170)."""
from .gshell_tets import GShell_Tets  # noqa: F401
from .hmsdf_tets_split import hmSDF_Tets  # noqa: F401
from .sdf_reg import compute_sdf_reg_loss  # noqa: F401
