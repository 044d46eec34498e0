"""Three and four heads on the tensor-core path, CPU side: dispatch, workspace layout and recompute chunking (no GPU)."""
import ctypes

import pytest

import enf_pde_b200 as E
from enf_pde_b200 import _lib

NEW_SHAPES = [(64, 3), (64, 4), (128, 3), (128, 4), (32, 4)]
BASE = dict(B=8, C=1000, Z=32, L=16, O=1, Dx=2, invariant_kind=3, use_window=1, precision=1, flags=0)


def _desc(**kw):
    return _lib.EnfDesc(**{**BASE, **kw})


@pytest.mark.parametrize("d,H", NEW_SHAPES)
def test_new_head_counts_run_on_the_tensor_cores(d, H):
    assert _lib.dispatch(_desc(d=d, H=H)) == (True, True)
    assert _lib.dispatch(_desc(d=d, H=H, flags=_lib.FLAG_FORWARD_ONLY)) == (True, False)
    assert _lib.dispatch(_desc(d=d, H=H, precision=0)) == (False, False)


@pytest.mark.parametrize("H", [1, 2, 3, 4])
def test_d16_stays_on_the_fp32_kernels(H):
    assert _lib.dispatch(_desc(d=16, H=H)) == (False, False)


@pytest.mark.parametrize("d,H", NEW_SHAPES)
def test_new_head_counts_get_the_tensor_core_workspace(d, H):
    """the logits, the operand stash and the hand-over buffer dthat (one per field chunk, summed over the head groups in place)."""
    lib = E.load_library()
    desc = _desc(d=d, H=H)
    assert lib.enf_xattn_workspace_bytes(ctypes.byref(desc)) > 0
    n = ctypes.c_int64(0)
    Cpad = (BASE["C"] + 127) // 128 * 128
    for name, size in (("slog", BASE["B"] * BASE["C"] * BASE["Z"] * H), ("that_img", BASE["B"] * BASE["Z"] * Cpad * max(d, 64) // 2),
                       ("dthat", BASE["B"] * BASE["Z"] * Cpad * d // 2)):
        assert lib.enf_debug_ws_offset(ctypes.byref(desc), name.encode(), ctypes.byref(n)) >= 0, name
        assert n.value == size, (name, n.value, size)
    fp32 = _desc(d=d, H=H, precision=0)
    assert lib.enf_debug_ws_offset(ctypes.byref(fp32), b"dthat", ctypes.byref(n)) < 0


@pytest.mark.parametrize("d,H", NEW_SHAPES)
def test_new_head_counts_chunk_in_recompute_mode(d, H):
    lib = E.load_library()
    size = lambda **o: lib.enf_xattn_workspace_bytes(ctypes.byref(_desc(d=d, H=H, **o)))
    stash = size()
    one = size(flags=_lib.FLAG_RECOMPUTE, chunk_fields=1)
    assert one < size(flags=_lib.FLAG_RECOMPUTE, chunk_fields=2) < stash
    assert size(flags=_lib.FLAG_RECOMPUTE, chunk_fields=BASE["B"]) == stash
    cap = (one + stash) // 2
    n = lib.enf_xattn_chunk_for_cap(ctypes.byref(_desc(d=d, H=H)), cap)
    assert 1 <= n < BASE["B"] and size(flags=_lib.FLAG_RECOMPUTE, chunk_fields=n) <= cap
    assert size(flags=_lib.FLAG_RECOMPUTE, chunk_fields=n + 1) > cap
