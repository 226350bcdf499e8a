"""The Chamfer normal / Laplacian term entry points: exported, workspace formula, and bad arguments rejected on the host, with a
negative status and a message, before any launch (no device needed)."""
import ctypes

import numpy as np

from geniconet_b200 import _lib

L = _lib.lib
ARG = -1
P = 1 << 12                        # a non-null dummy pointer: every call below fails before it is dereferenced
LEVEL = 2
V = 10 * 4 ** LEVEL + 2
PLAN = _lib.plan_blob(_lib.PLAN_LOSS, LEVEL)


def _args(**kw):
    a = dict(plan_host=PLAN.ctypes.data, plan_dev=P, v=P, tn=P, tnsb=60, tnsn=3, tnsc=1, tl=P, tlsb=60, tlsn=3, tlsc=1,
             idx_xy=P, idx_yx=P)
    a.update(kw)
    return a


def _fwd(out=P, ws=P, B=2, M=20, **kw):
    return L.gin_chamfer_terms_fwd(*_args(**kw).values(), out, ws, B, M, None)


def _bwd(dout=P, dv=P, ws=P, B=2, M=20, **kw):
    return L.gin_chamfer_terms_bwd(*_args(**kw).values(), dout, dv, ws, B, M, None)


def test_chamfer_terms_symbols_are_exported():
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for n in ('gin_chamfer_terms_ws_bytes', 'gin_chamfer_terms_fwd', 'gin_chamfer_terms_bwd'):
        assert hasattr(lib, n) and n in _lib.EXPORTS, n


def test_chamfer_terms_ws_bytes():
    # backward: g_n and g_L (12 B each) and two 32 B fixed-point accumulators per output vertex; forward: 1024 x 4 fp64 partials
    for B, level, M in ((36, 5, 10242), (1, 5, 100000), (4, 3, 7), (2, 1, 1)):
        bv = B * (10 * 4 ** level + 2)
        assert L.gin_chamfer_terms_ws_bytes(B, level, M) == max(bv * 88, 1024 * 4 * 8), (B, level, M)
    assert L.gin_chamfer_terms_ws_bytes(1, 0, 5) == 1024 * 4 * 8
    # the gin_ring_ops_bwd workspace fits in the accumulators it reuses
    assert L.gin_ring_ops_ws_bytes(36, 5) <= 36 * (10 * 4 ** 5 + 2) * 64
    for args in ((0, 5, 5), (-1, 5, 5), (2, -1, 5), (2, 10, 5), (2, 5, 0)):
        assert L.gin_chamfer_terms_ws_bytes(*args) == 0, args


def _rejects(call, *words, **kw):
    assert call(**kw) == ARG, kw
    msg = L.gin_last_error()
    for w in words:
        assert w in msg, (kw, msg)


def test_chamfer_terms_fwd_rejects_bad_arguments():
    assert _fwd(plan_host=None) < 0 and b'plan' in L.gin_last_error()
    assert _fwd(plan_dev=None) == ARG and b'plan' in L.gin_last_error()
    for k in ('v', 'ws'):
        _rejects(_fwd, b'null', **{k: None})
    _rejects(_fwd, b'null', out=None)
    _rejects(_fwd, b'null', b'normals', tn=None, tl=None)
    _rejects(_fwd, b'null', b'direction', idx_xy=None, idx_yx=None)
    _rejects(_fwd, b'negative', B=-1)
    _rejects(_fwd, b'M=0', M=0)
    _rejects(_fwd, b'M=-3', M=-3)
    _rejects(_fwd, b'2^31', B=30000, M=100000)
    bad = PLAN.copy()
    bad[2] = 12                                                 # GinLossPlanHdr.level
    _rejects(_fwd, b'level', plan_host=bad.ctypes.data)
    other = _lib.plan_blob(_lib.PLAN_HEXCONV, LEVEL)
    assert _fwd(plan_host=other.ctypes.data) < 0 and b'loss plan' in L.gin_last_error()
    # one term and one direction are enough to pass the checks; an empty batch is a no-op
    assert _fwd(B=0, v=None, out=None, ws=None, tn=None, idx_yx=None) == 0


def test_chamfer_terms_bwd_rejects_bad_arguments():
    for k in ('v', 'ws'):
        _rejects(_bwd, b'null', **{k: None})
    _rejects(_bwd, b'null', dv=None)
    _rejects(_bwd, b'dout', dout=None)
    _rejects(_bwd, b'null', tn=None, tl=None)
    _rejects(_bwd, b'null', idx_xy=None, idx_yx=None)
    _rejects(_bwd, b'negative', B=-2)
    _rejects(_bwd, b'M=0', M=0)
    bad = PLAN.copy()
    bad[2] = -1
    _rejects(_bwd, b'level', plan_host=bad.ctypes.data)
    assert _bwd(B=0, v=None, dv=None, ws=None, dout=None) == 0
    assert isinstance(V, int) and np.int32(PLAN[4]) == V       # the header field the entry points read V from
