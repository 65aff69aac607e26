"""lasgun_b200 — B200-native per-pixel render loop of nfrasser/lasgun behind the
reference's scene-builder / capture API (see DESIGN.md)."""
from .api import Aggregate, Camera, Film, Material, ObjData, ObjRef, Scene, parse_obj_text  # noqa: F401
from .render import Accel, capture, capture_guides, capture_linear, capture_subset, render  # noqa: F401
