"""CPU: the attention-dropout mask of the oracle (numpy Philox4x32-10) and argument checks of the dropout entry points,
without a GPU."""
import ctypes

import numpy as np
import pytest

from llamax_b200 import _lib
from tests import attention_dropout_ref as DR


@pytest.mark.parametrize("ctr,key,want", [
    ([0, 0, 0, 0], [0, 0], "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
    ([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2, "408f276d 41c83b0e a20bc7c6 6d5451fd"),
    ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0], "d16cfe09 94fdcceb 5001e420 24126ea1"),
])
def test_philox_known_answers(ctr, key, want):
    got = DR.philox4x32_10(np.array(ctr, dtype=np.uint64), np.array(key, dtype=np.uint64))
    assert " ".join(f"{int(w):08x}" for w in got) == want


@pytest.mark.parametrize("p", [0.1, 0.5, 0.9])
def test_keep_fraction(p):
    t, scale = DR.attention_dropout_threshold(p)
    assert scale == 256.0 / (256 - t)
    keep = DR.attention_dropout_keep(0x0123456789ABCDEF, 8, 2, 4, 512, p)   # 2M decisions
    n = keep.numel()
    f = 1 - t / 256
    assert abs(keep.float().mean().item() - f) <= 5 * (f * (1 - f) / n) ** 0.5


def test_keep_mask_layout():
    """A window is the matching slice of the whole mask; the counter's words select distinct masks."""
    seed, S = (1 << 40) + 12345, 300
    full = DR.attention_dropout_keep(seed, 4 * 7, 2, 3, S, 0.5)
    win = DR.attention_dropout_keep(seed, 4 * 7, 2, 3, S, 0.5, q_start=37, q_len=100, kv_start=21, kv_len=201)
    assert win.equal(full[:, :, 37:137, 21:222])
    assert not full[0, 0].equal(full[0, 1]) and not full[0, 0].equal(full[1, 0])      # b * Hq + hq
    assert not full.equal(DR.attention_dropout_keep(seed, 4 * 8, 2, 3, S, 0.5))         # offset / 4
    assert not full.equal(DR.attention_dropout_keep(seed + (1 << 32), 4 * 7, 2, 3, S, 0.5))   # high key word
    assert DR.attention_dropout_keep(seed, 4 * 7, 1, 1, 64, 0.001).all()               # t = 0: nothing dropped
    assert DR.attention_dropout_threshold(0.999) == (256, 0.0)


def _ptr():
    buf = ctypes.create_string_buffer(4096)
    return buf, ctypes.cast(buf, ctypes.c_void_p)


def _fwd(lib, p, D=128, dropout_p=0.1, null_q=False):
    return lib.llamax_attn_fwd_dropout(None if null_q else p, 128, p, 128, p, 128, p, 128, p, 1, 16, 1, 1, D, 0, None,
                                       None, 1.0, dropout_p, 1, 0, None)


def _bwd(lib, p, D=128, dropout_p=0.1, null_q=False):
    return lib.llamax_attn_bwd_dropout(None if null_q else p, 128, p, 128, p, 128, p, 128, p, p, 128, p, 128, p, 128,
                                       p, 128, p, p, 1, 16, 1, 1, D, 0, None, None, None, 1.0, None, dropout_p, 1, 0,
                                       None)


def _bwd_det(lib, p, D=128, dropout_p=0.1, null_q=False):
    return lib.llamax_attn_bwd_deterministic_dropout(None if null_q else p, 128, p, 128, p, 128, p, 128, p, p, 128, p,
                                                     128, p, 128, p, 128, p, 1, 16, 1, 1, D, 0, None, None, None, 1.0,
                                                     None, dropout_p, 1, 0, None)


@pytest.mark.parametrize("call", [_fwd, _bwd, _bwd_det])
def test_dropout_entry_points_validate_arguments_without_gpu(call):
    import __graft_entry__ as g

    g.build()
    lib = _lib.load()
    buf, p = _ptr()
    assert call(lib, p, null_q=True) == -1 and b"null" in lib.llamax_last_error()
    for bad in (-0.1, 1.0, 1.5, float("nan")):
        assert call(lib, p, dropout_p=bad) == -1 and b"dropout_p" in lib.llamax_last_error()
    assert call(lib, p, D=32) == -1 and b"head_dim" in lib.llamax_last_error()
