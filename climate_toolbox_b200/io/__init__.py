from .io import standardize_climate_data, load_bcsd  # noqa: F401  (reference io/__init__.py:1)
from .io import decode_packed  # noqa: F401
