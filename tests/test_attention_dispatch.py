"""Window-attention forward kernel choice (host arithmetic in the C-ABI library, no GPU): every window of 16 or more tokens
gets a tcgen05 kernel (attn_tc3.cu or attn_tc2.cu, which also write the row statistics lse), smaller ones the mma.sync fallback."""
import itertools
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


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


@pytest.mark.parametrize("window", [(8, 7, 7), (8, 12, 12), (1, 7, 7), (1, 12, 12)])
def test_every_window_of_16_tokens_gets_a_tcgen05_kernel(K, window):
    L = (2 * window[0] - 1) * (2 * window[1] - 1) * (2 * window[2] - 1)
    prev = K.set_attention_impl("auto")
    try:
        for impl in ("auto", "tc2", "tc3"):
            K.set_attention_impl(impl)
            for eff in itertools.product(*(range(1, w + 1) for w in window)):
                for shifted in (False, True):
                    g = _geometry(window, eff, shifted)
                    for nH in (4, 32):
                        has_lse = K.window_attention_has_lse(torch.empty(nH, L), g)
                        assert has_lse == (g.N >= 16), f"{impl}: window {window}, effective {eff}, shifted {shifted}, nH {nH}"
    finally:
        K.set_attention_impl(prev)


def test_attention_impl_selector(K):
    prev = K.set_attention_impl("tc2")
    try:
        assert K.set_attention_impl("tc3") == "tc2"
        assert K.set_attention_impl("auto") == "tc3"
        for retired in ("mma", "tc1"):
            with pytest.raises(K.LavtError):
                K.set_attention_impl(retired)
        lib = K.lib()
        for code in (1, 2, 5, -1):          # retired and unknown codes select auto
            lib.lavt_set_attention_impl(3)
            assert lib.lavt_set_attention_impl(code) == 3
            assert lib.lavt_set_attention_impl(0) == 0
    finally:
        K.set_attention_impl(prev)
