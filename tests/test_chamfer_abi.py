"""The Chamfer entry points: exported, workspace formula, and bad arguments rejected on the host, with a negative status and a
message, before any launch (no device needed)."""
import ctypes

from geniconet_b200 import _lib

L = _lib.lib
ARG = -1
P = 1 << 12                        # a non-null dummy pointer: every call below fails before it is dereferenced


def _fwd(**kw):
    a = dict(x=P, xsb=30, xsn=3, xsc=1, y=P, ysb=15, ysn=3, ysc=1, d_xy=P, idx_xy=P, d_yx=P, idx_yx=P, ws=P, B=2, N=10, M=5)
    a.update(kw)
    return L.gin_chamfer_fwd(*a.values(), None)


def _bwd(**kw):
    a = dict(x=P, xsb=30, xsn=3, xsc=1, y=P, ysb=15, ysn=3, ysc=1, idx_xy=P, g_xy=P, idx_yx=P, g_yx=P, dx=P, dy=P, ws=P, B=2, N=10, M=5)
    a.update(kw)
    return L.gin_chamfer_bwd(*a.values(), None)


def test_chamfer_symbols_are_exported():
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for n in ('gin_chamfer_ws_bytes', 'gin_chamfer_fwd', 'gin_chamfer_bwd'):
        assert hasattr(lib, n) and n in _lib.EXPORTS, n


def test_chamfer_ws_bytes():
    # 32 B per point of the larger set: int64 fixed-point sums [3], exponent, count (backward); covers the forward's 64-bit keys
    assert L.gin_chamfer_ws_bytes(36, 10242, 10242) == 36 * 10242 * 32
    assert L.gin_chamfer_ws_bytes(1, 10242, 100000) == 100000 * 32
    assert L.gin_chamfer_ws_bytes(4, 37, 5) == 4 * 37 * 32 >= 8 * 4 * (37 + 5)
    for args in ((0, 5, 5), (2, 0, 5), (2, 5, 0), (-1, 5, 5)):
        assert L.gin_chamfer_ws_bytes(*args) == 0, args


def test_chamfer_fwd_rejects_bad_arguments():
    for k in ('x', 'y', 'ws'):
        assert _fwd(**{k: None}) == ARG and b'null' in L.gin_last_error(), k
    assert _fwd(d_xy=None, idx_xy=None, d_yx=None, idx_yx=None) == ARG and b'null' in L.gin_last_error()
    assert _fwd(d_xy=None) == ARG and b'index' in L.gin_last_error()       # an index output needs its distance output
    assert _fwd(d_yx=None) == ARG
    assert _fwd(B=-1) == ARG and b'negative' in L.gin_last_error()
    assert _fwd(N=0) == ARG and b'empty' in L.gin_last_error()
    assert _fwd(M=0) == ARG and _fwd(N=-3) == ARG
    assert _fwd(B=65536) == ARG and b'65535' in L.gin_last_error()
    assert _fwd(B=40000, N=60000) == ARG and b'2^31' in L.gin_last_error()
    assert _fwd(B=0, x=None, y=None, ws=None, d_xy=None, idx_xy=None, d_yx=None, idx_yx=None, N=0, M=0) == 0   # empty batch: no-op


def test_chamfer_bwd_rejects_bad_arguments():
    for k in ('x', 'y', 'ws'):
        assert _bwd(**{k: None}) == ARG and b'null' in L.gin_last_error(), k
    assert _bwd(g_xy=None, g_yx=None) == ARG and b'cotangent' in L.gin_last_error()
    assert _bwd(idx_xy=None) == ARG and b'indices' in L.gin_last_error()  # a cotangent needs its indices
    assert _bwd(idx_yx=None) == ARG
    assert _bwd(dx=None, dy=None) == ARG
    assert _bwd(B=-2) == ARG and _bwd(N=0) == ARG and _bwd(M=0) == ARG
    assert _bwd(B=70000) == ARG
    assert _bwd(B=3, M=1 << 30) == ARG and b'2^31' in L.gin_last_error()
    assert _bwd(B=0, x=None, y=None, ws=None, idx_xy=None, g_xy=None, idx_yx=None, g_yx=None, dx=None, dy=None) == 0
