"""CPU: cn_gru_gates_backward_pairs refuses bad arguments before it touches a device (pure host checks: the pointers below
are never dereferenced), so a caller's mistake is an error message rather than a fault on the GPU."""
import ctypes as C

import pytest

from crowdnav_dsrnn_b200 import _lib

BASE = 1 << 24                  # 256-byte aligned fake device addresses; nothing is launched for any call below
GOOD = dict(grad_h=BASE, d=BASE + 0x10000, d_live=1, m_next=BASE + 0x20000, ws=BASE + 0x30000, h_prev=BASE + 0x40000,
            m_cur=BASE + 0x50000, g_hi=BASE + 0x60000, g_lo=BASE + 0x70000, rows=77, hid=256)
ORDER = ("grad_h", "d", "d_live", "m_next", "ws", "h_prev", "m_cur", "g_hi", "g_lo", "rows", "hid")
INTS = ("d_live", "rows", "hid")

BAD = [
    ("rows 0", dict(rows=0)),
    ("rows negative", dict(rows=-3)),
    ("hid not a multiple of 4", dict(hid=6)),
    ("hid 0", dict(hid=0)),
    ("live d without m_next", dict(m_next=None)),
    ("h_prev without m_cur", dict(m_cur=None)),
    ("grad_h misaligned", dict(grad_h=BASE + 4)),
    ("d misaligned", dict(d=BASE + 0x10000 + 8)),
    ("ws misaligned", dict(ws=BASE + 0x30000 + 4)),
    ("h_prev misaligned", dict(h_prev=BASE + 0x40000 + 12)),
    ("g_hi misaligned", dict(g_hi=BASE + 0x60000 + 2)),
    ("g_lo misaligned", dict(g_lo=BASE + 0x70000 + 4)),
    ("grad_h NULL", dict(grad_h=None)),
    ("d NULL", dict(d=None)),
    ("ws NULL", dict(ws=None)),
    ("g_hi NULL", dict(g_hi=None)),
    ("g_lo NULL", dict(g_lo=None)),
]


@pytest.mark.parametrize("what,change", BAD, ids=[b[0] for b in BAD])
def test_gru_gates_backward_pairs_refuses_bad_arguments(what, change):
    lib = _lib.load()
    args = dict(GOOD, **change)
    call = [args[k] if k in INTS else (C.c_void_p(args[k]) if args[k] is not None else None) for k in ORDER]
    assert lib.cn_gru_gates_backward_pairs(*call, None) != 0, what
    assert b"cn_gru_gates_backward_pairs" in lib.cn_last_error()
