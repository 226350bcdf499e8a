"""The synchronised-BatchNorm entry points are exported and reject bad arguments on the host, with a negative status, before any launch."""
from geniconet_b200 import _lib

L = _lib.lib
ARG = -1

NEW = ('gin_bn_sync_record_bytes', 'gin_bn_sync_stats_total', 'gin_bn_sync_stats_total_from_parts', 'gin_bn_sync_stats_final',
       'gin_bn_sync_bwd_reduce', 'gin_bn_sync_bwd_reduce_pair', 'gin_bn_sync_bwd_final', 'gin_bn_bwd_apply', 'gin_bn_bwd_apply_pair')


def test_exported():
    for name in NEW:
        assert name in _lib.EXPORTS and hasattr(L, name), name


def test_record_bytes():
    assert L.gin_bn_sync_record_bytes(64, 0) == 8 * (2 * 64 + 1)
    assert L.gin_bn_sync_record_bytes(64, 1) == 2 * 8 * (2 * 64 + 1)          # a pair: A's record, then B's
    assert L.gin_bn_sync_record_bytes(0, 0) == 0


def _total(**kw):
    a = dict(y=1, ld=64, rows=100, C=64, rec=1, ws=1)
    a.update(kw)
    return L.gin_bn_sync_stats_total(*a.values(), None)


def _total_parts(**kw):
    a = dict(parts=1, nparts=4, ld=128, rows=100, C=64, colA=0, colB=64, rec=1)
    a.update(kw)
    return L.gin_bn_sync_stats_total_from_parts(*a.values(), None)


def _final(**kw):
    a = dict(recs=1, world=2, C=64, gA=1, bA=1, epsA=1e-5, momA=0.1, rmA=1, rvA=1, nbA=1, statA=1,
             gB=None, bB=None, epsB=0.0, momB=0.0, rmB=None, rvB=None, nbB=None, statB=None)
    a.update(kw)
    return L.gin_bn_sync_stats_final(*a.values(), None)


def _reduce(**kw):
    a = dict(dout=1, ldg=64, mask=1, y=1, ld=64, y_fp16=1, stat=1, rec=1, ws=1, B=2, level=3, C=64, relu_from_y=1)
    a.update(kw)
    return L.gin_bn_sync_bwd_reduce(*a.values(), None)


def _reduce_pair(**kw):
    a = dict(dout=1, ldg=64, mask=1, yA=1, ldA=64, statA=1, yB=1, ldB=128, statB=1, y_fp16=1, rec=1, ws=1, B=2, level=3, C=64, relu_from_y=1)
    a.update(kw)
    return L.gin_bn_sync_bwd_reduce_pair(*a.values(), None)


def _bwd_final(**kw):
    a = dict(recs=1, world=2, rank=1, C=64, bstatA=1, bstatB=None)
    a.update(kw)
    return L.gin_bn_sync_bwd_final(*a.values(), None)


def _apply(**kw):
    a = dict(dout=1, ldg=64, mask=1, y=1, ld=64, y_fp16=1, stat=1, bstat=1, dy_b=1, ldo=64, dy_f=None, ldf=0, B=2, level=3, C=64, relu_from_y=1)
    a.update(kw)
    return L.gin_bn_bwd_apply(*a.values(), None)


def _apply_pair(**kw):
    a = dict(dout=1, ldg=64, mask=1, yA=1, ldA=64, statA=1, bstatA=1, dyA=1, ldoA=64, yB=1, ldB=128, statB=1, bstatB=1, dyB=1, ldoB=128,
             y_fp16=1, B=2, level=3, C=64, relu_from_y=1)
    a.update(kw)
    return L.gin_bn_bwd_apply_pair(*a.values(), None)


def test_stats_total_rejects_bad_arguments():
    for k in ('y', 'rec', 'ws'):
        assert _total(**{k: None}) == ARG, k
    assert _total(rows=0) == ARG
    for C in (0, 12, 24):                                                # C/8 must divide 256
        assert _total(C=C, ld=64) == ARG, C
    assert _total(ld=32) == ARG                                          # row stride below C
    assert _total(ld=66) == ARG                                          # not 16-byte aligned rows


def test_stats_total_from_parts_rejects_bad_arguments():
    for k in ('parts', 'rec'):
        assert _total_parts(**{k: None}) == ARG, k
    assert _total_parts(nparts=0) == ARG
    assert _total_parts(nparts=148 * 4 + 1) == ARG
    assert _total_parts(rows=-1) == ARG
    assert _total_parts(C=24) == ARG
    assert _total_parts(colA=-1) == ARG
    assert _total_parts(colB=-2) == ARG
    assert _total_parts(ld=100) == ARG                                   # column slice colB + C beyond the row
    assert _total_parts(ld=32, colB=-1) == ARG


def test_stats_final_rejects_bad_arguments():
    assert _final(recs=None) == ARG
    assert _final(statA=None) == ARG
    assert _final(world=0) == ARG
    assert _final(C=12) == ARG


def test_bwd_reduce_rejects_bad_arguments():
    for k in ('dout', 'y', 'stat', 'rec', 'ws'):
        assert _reduce(**{k: None}) == ARG, k
    assert _reduce(B=0) == ARG
    assert _reduce(level=10) == ARG
    assert _reduce(C=24) == ARG
    for k in ('dout', 'yA', 'yB', 'statA', 'statB', 'rec', 'ws'):
        assert _reduce_pair(**{k: None}) == ARG, k
    assert _reduce_pair(level=-1) == ARG
    assert _reduce_pair(C=0) == ARG


def test_bwd_final_rejects_bad_arguments():
    for k in ('recs', 'bstatA'):
        assert _bwd_final(**{k: None}) == ARG, k
    assert _bwd_final(world=0, rank=0) == ARG
    assert _bwd_final(rank=2) == ARG                                     # rank outside the world
    assert _bwd_final(rank=-1) == ARG
    assert _bwd_final(C=96) == ARG


def test_bwd_apply_rejects_bad_arguments():
    for k in ('dout', 'y', 'stat', 'bstat'):
        assert _apply(**{k: None}) == ARG, k
    assert _apply(dy_b=None) == ARG                                      # no output at all
    assert _apply(B=0) == ARG
    assert _apply(C=40) == ARG
    for k in ('dout', 'yA', 'yB', 'statA', 'statB', 'bstatA', 'bstatB', 'dyA', 'dyB'):
        assert _apply_pair(**{k: None}) == ARG, k
    assert _apply_pair(level=10) == ARG
