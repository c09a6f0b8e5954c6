"""Model factories of the hot path (mirror of what /root/reference/models/__init__.py exports)."""
from .wrappers import BaseModel, StyleGAN, StyleGAN2, get_model, get_instrumented_model  # noqa: F401
