"""CPU-side checks (-m "not gpu") of the one-call batch-sharded step's symmetric InfoNCE branch: the workspace it plans and
the new C-ABI symbols.  (Planning is host-only arithmetic: no device is touched.)"""
import ctypes
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SYM, DOT, BILINEAR, FAST, STRICT = 3, 0, 1, 0, 1


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from mi_b200 import _lib
    return _lib.load()


@pytest.mark.parametrize("precision", [FAST, STRICT])
@pytest.mark.parametrize("critic", [DOT, BILINEAR])
@pytest.mark.parametrize("Bl,D", [(600, 72), (8192, 1024), (256, 64)])
def test_sharded_sym_workspace_covers_its_stages(lib, Bl, D, critic, precision):
    """non-zero for every world size 1-8 (it was 0 before the symmetric branch existed), and at least the larger of the
    statistics and gradient passes' own scratch plus the [B, D] fp32 dY contributions"""
    for world in range(1, 9):
        B = Bl * world
        got = lib.mi_sharded_critic_workspace_bytes(Bl, world, D, critic, SYM, precision)
        stages = max(lib.mi_score_stats_rc_workspace_bytes(Bl, B, D), lib.mi_score_grad_workspace_bytes(Bl, B, D, precision))
        assert got > 0, (world, Bl, D)
        assert got >= stages + B * D * 4, (world, got, stages)


def test_sharded_sym_workspace_rejects_bad_shapes(lib):
    assert lib.mi_sharded_critic_workspace_bytes(600, 2, 60, BILINEAR, SYM, FAST) == 0        # D % 8 != 0
    assert lib.mi_sharded_critic_workspace_bytes(0, 2, 64, BILINEAR, SYM, FAST) == 0
    assert lib.mi_sharded_critic_workspace_bytes(600, 2, 64, BILINEAR, SYM + 1, FAST) == 0


def test_merge_sym_scratch_and_new_symbols_exported(lib):
    from mi_b200 import _lib
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for n in ("mi_score_stats_rc_ex", "mi_merge_sym_stats", "mi_merge_sym_stats_scratch_doubles"):
        assert hasattr(raw, n) and n in _lib.PROTOTYPES
    assert lib.mi_merge_sym_stats_scratch_doubles(65536) >= 65536 // 256 + 16
    assert lib.mi_merge_sym_stats_scratch_doubles(1) >= 17
    assert lib.mi_merge_sym_stats_scratch_doubles(0) == 0


def test_stats_rc_ex_and_merge_reject_without_a_device(lib):
    """no CPU fallback: on a machine without an sm_100 device both new entry points fail before touching memory"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("checks the no-GPU failure mode")
    st = lib.mi_merge_sym_stats(None, None, 0, 1, 1, None, None, None, None)
    assert st != 0
    st = lib.mi_score_stats_rc_ex(None, 64, 1, None, 64, 1, None, None, 0, 256, 512, 64, 1.0, None, None, None, None, 0, 0,
                                  None, 0, None)
    assert st != 0
