"""mutual-information-multimodal_b200 — B200-native (sm_100a) MI critic / estimator hot path.

Importable as ``mi_b200`` (see ``/mi_b200.py`` at the repo root; the directory name carries a
hyphen).  Layout:

  csrc/        hand-written CUDA (tcgen05 / TMEM / TMA tile engine) + the C ABI (include/mi_b200.h)
  _lib.py      ctypes binding of libmi_b200.so (built in-tree by ``__graft_entry__.build()``)
  ops.py       stage-level wrappers on torch tensors (device memory and streams only)
  critic.py    host-side mirror of the reference API: create_mi_pairs / FusedCritic /
               dv_bound_loss / infonce_bound_loss (mutual_info_img_txt/mi_critics.py, main_utils.py:80-110)
  validate.py  gdv_calculation (validate.py:16-49) on the same tile engine
  dist.py      batch-sharded multi-GPU path (torch.distributed all-gathers + scalar reductions)

There is no CPU fallback: every compute entry point raises when the CUDA library or a Blackwell
device is missing.
"""
from . import _lib  # noqa: F401
from .critic import (  # noqa: F401
    FusedCritic, FusedMLPCritic, PairBatch, ScoreHandle, create_mi_pairs, create_mi_pairs_tensor, dv_bound_loss, infonce_bound_loss,
    js_bound_loss, mi_estimator_loss, nwj_bound_loss, select_estimator, sharded_mi_loss,
)
from .ops import MIError  # noqa: F401
from .validate import gdv_calculation, gdv_terms  # noqa: F401

__all__ = [
    "FusedCritic", "FusedMLPCritic", "PairBatch", "ScoreHandle", "create_mi_pairs", "create_mi_pairs_tensor", "dv_bound_loss",
    "infonce_bound_loss", "js_bound_loss", "nwj_bound_loss", "mi_estimator_loss", "select_estimator", "sharded_mi_loss", "MIError", "gdv_calculation", "gdv_terms",
]
