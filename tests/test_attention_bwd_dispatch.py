"""Window-attention backward kernel choice (host arithmetic in the C-ABI library, no GPU): every window of 16 or more tokens with the
forward's saved lse gets a kernel.  Full 7 x 7 windows with an even frame count keep attn_bwd_tc.cu, windows that fit the mma.sync kernel
keep it, and exactly the rest (full and large clamped 8 x 12 x 12 windows) go to attn_bwd_tc2.cu, the only kernel with a workspace."""
import itertools
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WINDOWS = [(8, 7, 7), (8, 12, 12), (1, 7, 7), (1, 12, 12)]


@pytest.fixture(scope="module")
def K():
    from lavt_rs_b200.build import build_library
    build_library()
    from lavt_rs_b200 import _cabi
    _cabi.lib()
    return _cabi


def _geometry(window, eff, shifted):
    """A clip whose effective window is eff: an axis where eff is the full window gets twice its extent (not clamped, so it keeps
    its shift), any other axis is clamped to eff."""
    from lavt_rs_b200.geometry import window_geometry
    size = [2 * w if e == w else e for w, e in zip(window, eff)]
    g = window_geometry(1, *size, window, shifted, True)
    assert (g.wd, g.wh, g.ww) == tuple(eff)
    return g


def _table_len(window):
    return (2 * window[0] - 1) * (2 * window[1] - 1) * (2 * window[2] - 1)


def _mma_fits(N, L):
    """shared memory of the mma.sync kernel (attn_bwd.cu): Q / K / V / dO (64 B per token each), a 16-byte token record, 3 table copies"""
    NP = (N + 15) // 16 * 16
    return NP * 272 + L * 12 + 32 <= 227 * 1024


def _sweep(window):
    for eff in itertools.product(*(range(1, w + 1) for w in window)):
        for shifted in (False, True):
            g = _geometry(window, eff, shifted)
            for nH in (4, 32):
                yield eff, shifted, nH, g


@pytest.mark.parametrize("window", WINDOWS)
def test_every_window_of_16_tokens_gets_a_backward_kernel(K, window):
    L = _table_len(window)
    prev = K.set_attention_bwd_impl("auto")
    try:
        for eff, shifted, nH, g in _sweep(window):
            t = torch.empty(nH, L)
            k = K.window_attention_bwd_kernel(t, g, has_lse=True)
            where = f"window {window}, effective {eff}, shifted {shifted}, nH {nH}: {k}"
            full7 = eff[1:] == (7, 7) and window[1:] == (7, 7) and eff[0] % 2 == 0 and window[0] == 8
            if g.N >= 16:
                assert k is not None, where
            if full7:
                assert k == "tc", where
            elif _mma_fits(g.N, L):
                assert k == "mma", where
            else:
                assert k == "tc2" and g.N <= 1152, where
            ws = K.window_attention_bwd_workspace_floats(t, g)
            if k != "tc2":
                assert ws == 0, where
            elif g.N > 128:
                assert ws >= (g.N + 127) // 128 * 128 * 32, where
            # without lse only the mma.sync kernel applies: the choice for shapes that fit it does not change
            k0 = K.window_attention_bwd_kernel(t, g, has_lse=False)
            assert k0 == ("mma" if _mma_fits(g.N, L) else None), where
    finally:
        K.set_attention_bwd_impl(prev)


def test_w12_windows_that_did_not_train_get_tc2(K):
    """The 8 x 12 x 12 windows that no backward kernel could run before: N = 1152, 576 and clamped 800 / 648."""
    L = _table_len((8, 12, 12))
    for eff in ((8, 12, 12), (4, 12, 12), (8, 10, 10), (8, 9, 9)):
        for shifted in (False, True):
            g = _geometry((8, 12, 12), eff, shifted)
            assert K.window_attention_bwd_kernel(torch.empty(4, L), g) == "tc2", eff


@pytest.mark.parametrize("window", WINDOWS)
def test_forced_tc2_applies_to_every_window_of_16_to_1152_tokens(K, window):
    L = _table_len(window)
    prev = K.set_attention_bwd_impl("tc2")
    try:
        for eff, shifted, nH, g in _sweep(window):
            t = torch.empty(nH, L)
            k = K.window_attention_bwd_kernel(t, g, has_lse=True)
            assert k == ("tc2" if g.N >= 16 else "mma"), f"window {window}, effective {eff}, shifted {shifted}, nH {nH}: {k}"
    finally:
        K.set_attention_bwd_impl(prev)


def test_mma_only_selection_keeps_its_meaning(K):
    L = _table_len((8, 12, 12))
    prev = K.set_attention_bwd_impl("mma")
    try:
        t = torch.empty(4, L)
        assert K.window_attention_bwd_kernel(t, _geometry((8, 12, 12), (8, 12, 12), True)) is None
        assert K.window_attention_bwd_kernel(t, _geometry((8, 12, 12), (2, 12, 12), True)) == "mma"
        t7 = torch.empty(4, _table_len((8, 7, 7)))
        assert K.window_attention_bwd_kernel(t7, _geometry((8, 7, 7), (8, 7, 7), True)) == "mma"
    finally:
        K.set_attention_bwd_impl(prev)


def test_attention_bwd_impl_selector(K):
    prev = K.set_attention_bwd_impl("tc2")
    try:
        assert K.set_attention_bwd_impl("mma") == "tc2"
        assert K.set_attention_bwd_impl("tc") == "mma"
        assert K.set_attention_bwd_impl("auto") == "tc"
        with pytest.raises(K.LavtError):
            K.set_attention_bwd_impl("tc3")
        lib = K.lib()
        for code, name in enumerate(("auto", "mma", "tc", "tc2")):
            lib.lavt_set_attention_bwd_impl(code)
            assert K.set_attention_bwd_impl("auto") == name
        for code in (4, 5, -1):              # unknown codes select auto
            lib.lavt_set_attention_bwd_impl(3)
            assert lib.lavt_set_attention_bwd_impl(code) == 3
            assert lib.lavt_set_attention_bwd_impl(0) == 0
        assert K.ATTN_BWD_KERNELS == {0: None, 1: "mma", 2: "tc", 3: "tc2"}
    finally:
        K.set_attention_bwd_impl(prev)
