"""B200-native BASD distillation-loss hot path (drop-in for the reference's `src/losses`).

Importable name: `vit_bias_aware_structural_distillation_b200` (the hyphenated spelling
`vit-bias-aware-structural-distillation_b200/` at the repo root is a symlink to this directory — hyphens are not
valid in Python module names)."""
from ._lib import BasdError, LIB_PATH, load  # noqa: F401
from .loss import (BASDLoss, GrassmannianLayerSelector, HostStager, align_token_count, cls_attention_rows,  # noqa: F401
                   geometric_relational_loss, marchenko_pastur_rank, query_mean_attention, workspace_view)

__all__ = ["BASDLoss", "GrassmannianLayerSelector", "HostStager", "align_token_count", "cls_attention_rows", "geometric_relational_loss",
           "marchenko_pastur_rank", "query_mean_attention", "BasdError", "load", "LIB_PATH", "workspace_view"]
