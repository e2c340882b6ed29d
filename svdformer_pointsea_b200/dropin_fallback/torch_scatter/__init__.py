"""Drop-in for torch_scatter as PointSea uses it (models_PointSea/mv_utils_zs.py:1,130: scatter(..., reduce="max")).

This directory is appended to sys.path (DROPIN_FALLBACK_PATH), so an installed torch_scatter is found first and this
package only when none is installed."""
from svdformer_pointsea_b200.scatter import scatter  # noqa: F401
