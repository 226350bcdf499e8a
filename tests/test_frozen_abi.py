"""The eval-mode BatchNorm backward entry points reject bad arguments on the host, with a negative status, before any launch."""
from geniconet_b200 import _lib

L = _lib.lib
ARG = -1


def _single(**kw):
    a = dict(dout=1, ldg=64, mask=None, y=1, ld=64, y_fp16=1, stat=1, bsum=None, dy_b=1, ldo=64, dy_f=None, ldf=0, ws=None, B=2, level=3,
             C=64, relu_from_y=1)
    a.update(kw)
    return L.gin_bn_eval_bwd(*a.values(), None)


def _pair(**kw):
    a = dict(dout=1, ldg=64, mask=None, yA=1, ldA=64, statA=1, bsumA=None, dyA=1, ldoA=64, yB=1, ldB=128, statB=1, bsumB=None, dyB=1,
             ldoB=128, y_fp16=1, ws=None, B=2, level=3, C=64, relu_from_y=1)
    a.update(kw)
    return L.gin_bn_eval_bwd_pair(*a.values(), None)


def test_eval_bwd_ws_bytes():
    assert L.gin_bn_eval_bwd_ws_bytes(64) == L.gin_bn_pair_ws_bytes(64) // 4 * 3
    assert L.gin_bn_eval_bwd_ws_bytes(0) == 0


def test_eval_bwd_rejects_bad_arguments():
    for k in ('dout', 'y', 'stat'):
        assert _single(**{k: None}) == ARG, k
    assert _single(dy_b=None) == ARG                                     # no output at all
    assert _single(bsum=1) == ARG                                        # sums need the workspace
    assert _single(B=0) == ARG
    assert _single(level=10) == ARG
    for C in (0, 12, 24, 512):                                           # C/8 must divide 256, and C <= 256
        assert _single(C=C, ldg=512, ld=512, ldo=512) == ARG, C
    assert _single(ldg=32) == ARG and b'stride' in L.gin_last_error()
    assert _single(ld=68) == ARG                                         # not a multiple of 8
    assert _single(ldo=32) == ARG
    assert _single(dy_f=1, ldf=60) == ARG


def test_eval_bwd_pair_rejects_bad_arguments():
    for k in ('dout', 'yA', 'yB', 'statA', 'statB', 'dyA', 'dyB'):
        assert _pair(**{k: None}) == ARG, k
    assert _pair(bsumA=1) == ARG and _pair(bsumB=1) == ARG               # sums need the workspace
    assert _pair(B=-1) == ARG
    assert _pair(C=96, ldg=96, ldA=96, ldB=192, ldoA=96, ldoB=192) == ARG
    assert _pair(C=512, ldg=512, ldA=512, ldB=1024, ldoA=512, ldoB=1024) == ARG
    assert _pair(ldB=32) == ARG and b'stride' in L.gin_last_error()
    assert _pair(ldoA=100) == ARG
